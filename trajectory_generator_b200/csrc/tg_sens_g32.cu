// Parameter-sensitivity kernels, 32 lanes per problem (see tg_kernels_sens.inc)
#define TG_GS 32
#define TG_SFX _g32
// fixed shapes (tg_shape.h) with instantiations in this translation unit: the ones tg_plan_polish gives 32 lanes
#define TG_SENS_FIXED TG_FIXED_CASE(TG_FIX_C3) TG_FIXED_CASE(TG_FIX_C4)
#include "tg_kernels_sens.inc"
