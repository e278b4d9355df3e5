// murty_ladder_kernel.cu -- the k-ladder instantiations of the two Murty kernel files (MurtyLadder, pda_internal.h):
// murty_ladder_kernel<R, FAST> and murty_cta_ladder_kernel<R>, with the launches that pick among them.  They live in a
// translation unit of their own because, compiled next to the plain kernels, they change the compiler's inlining
// decisions there (murty_cta_kernel<2> then calls its per-problem body instead of inlining it); apart, the plain
// kernels compile to the code they have without the ladder.
#undef PDA_CTA_PROFILE  // the profiling counters belong to the plain CTA kernel
#define PDA_MURTY_LADDER_TU
#include "murty_kernel.cu"
#include "murty_cta_kernel.cu"
