// M2 line-search kernels, 8 lanes per problem (see tg_kernels_solve.inc)
#define TG_GS 8
// the lock-step kernels run every warp through the same code at the same time: the block evaluators are inlined
#ifndef TG_NO_INLINE_LS
#define TG_INLINE_ALL
#endif
#define TG_SFX _g8
#define TG_LS_STAGE
// fixed shapes (tg_shape.h) with instantiations in this translation unit: the BASELINE configurations this group size serves
#define TG_LS_FIXED TG_FIXED_CASE(TG_FIX_C2) TG_FIXED_CASE(TG_FIX_C5A) TG_FIXED_CASE(TG_FIX_C5C)
#include "tg_kernels_solve.inc"
