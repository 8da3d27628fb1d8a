// Parameter-sensitivity kernels, 8 lanes per problem (see tg_kernels_sens.inc)
#define TG_GS 8
#define TG_SFX _g8
// fixed shapes (tg_shape.h) with instantiations in this translation unit: the ones tg_plan_polish gives 8 lanes
#define TG_SENS_FIXED TG_FIXED_CASE(TG_FIX_C2) TG_FIXED_CASE(TG_FIX_C5A) TG_FIXED_CASE(TG_FIX_C5C)
#include "tg_kernels_sens.inc"
