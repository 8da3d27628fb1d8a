// M2 QP-stage kernel with 64 lanes (two warps) per problem, for shapes with more than 32 variables: every
// lane-strided loop of the stage then takes one pass (see tg_kernels_solve.inc, tg_eval.h: TG_GS == 64)
#define TG_GS 64
#define TG_QP_STAGE
#define TG_SFX _g64
// fixed shapes (tg_shape.h) with instantiations in this translation unit: the BASELINE configurations this group size serves
#define TG_QP_FIXED TG_FIXED_CASE(TG_FIX_C3)
#include "tg_kernels_solve.inc"
