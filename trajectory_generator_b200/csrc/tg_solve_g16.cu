// M2 line-search and QP-stage kernels, 16 lanes per problem (see tg_kernels_solve.inc)
#define TG_GS 16
// the lock-step kernels run every warp through the same code at the same time: the block evaluators are inlined
#ifndef TG_NO_INLINE_LS
#define TG_INLINE_ALL
#endif
#define TG_SFX _g16
#define TG_LS_STAGE
#define TG_QP_STAGE
// fixed shapes (tg_shape.h) with instantiations in this translation unit: the BASELINE configurations this group size serves
#define TG_LS_FIXED TG_FIXED_CASE(TG_FIX_C3) TG_FIXED_CASE(TG_FIX_C4)
// QP stage: the shapes whose subproblem has at most 16 variables once the terminal location rows are eliminated (tg_sqp_qp_dim)
#define TG_QP_FIXED TG_FIXED_CASE(TG_FIX_C5A) TG_FIXED_CASE(TG_FIX_C5C)
#include "tg_kernels_solve.inc"
