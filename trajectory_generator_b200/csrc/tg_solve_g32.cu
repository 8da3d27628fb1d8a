// M2 solve kernels, 32 lanes per problem (see tg_kernels_solve.inc): begin, line search, QP stage, finish
#define TG_GS 32
// the lock-step kernels run every warp through the same code at the same time: the block evaluators are inlined
#ifndef TG_NO_INLINE_LS
#define TG_INLINE_ALL
#endif
#define TG_SFX _g32
#define TG_LS_STAGE
#define TG_QP_STAGE
// QP stage: 5 CTAs (20 warps) per SM at <= 96 registers -- the staged state without the factor L leaves room for them in
// shared memory (C2 / C5: QP stage -4 ... -8 %; the 64-lane kernels of tg_solve_g64.cu lose 5 % at 96 registers and keep 4)
#define TG_QP_MIN_CTAS 5
// fixed shapes (tg_shape.h) with instantiations in this translation unit: the BASELINE configurations this group size serves
#define TG_QP_FIXED TG_FIXED_CASE(TG_FIX_C2) TG_FIXED_CASE(TG_FIX_C4)
#include "tg_kernels_solve.inc"
