// risp_fused.cu's step on crops of a store of 8-bit raw codes (fused_step_store_u8_launch), in an object of its own: see the
// note above fused_handles there.  A non-template kernel has external linkage, so this object's preparation kernel is renamed.
#define RISP_FUSED_PART 3
#define fused_prep_kernel fused_store_u8_prep_kernel
#include "risp_fused.cu"
