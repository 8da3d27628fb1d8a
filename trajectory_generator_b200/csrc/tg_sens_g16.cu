// Parameter-sensitivity kernels, 16 lanes per problem (see tg_kernels_sens.inc)
#define TG_GS 16
#define TG_SFX _g16
#include "tg_kernels_sens.inc"
