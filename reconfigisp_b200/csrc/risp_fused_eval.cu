// risp_fused.cu's evaluation entry points (fused_eval_launch, fused_eval_store_launch), in an object of their own: see the
// note above fused_handles there.  A non-template kernel has external linkage, so this object's preparation kernel is renamed.
#define RISP_FUSED_PART 1
#define fused_prep_kernel fused_eval_prep_kernel
#include "risp_fused.cu"
