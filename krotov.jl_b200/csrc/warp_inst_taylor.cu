// krotov_warp_kernel instances with the truncated-Taylor step (prop_method=Expmv), one warp per trajectory (d <= 32).
#include "kernel_table.h"
namespace kr {
void add_warp_instances_taylor(KernelMap &t, KernelMap &emul) {
    // runtime L, rows reloaded from L1/L2 per use: the W set of the Chebyshev runtime family
    KR_INSTT(1, 0, 512); KR_INSTT(2, 0, 512); KR_INSTT(3, 0, 512); KR_INSTT(4, 0, 512); KR_INSTT(5, 0, 512);
    KR_INSTT(6, 0, 512); KR_INSTT(7, 0, 512); KR_INSTT(8, 0, 512); KR_INSTT(10, 0, 512); KR_INSTT(12, 0, 512);
    KR_INSTT(16, 0, 256); KR_INSTT(20, 0, 256); KR_INSTT(24, 0, 256); KR_INSTT(31, 0, 256);
    // register-resident term rows, one and two controls
    KR_INSTT(1, 1, 256); KR_INSTT(2, 1, 256); KR_INSTT(3, 1, 256); KR_INSTT(4, 1, 256); KR_INSTT(6, 1, 256); KR_INSTT(8, 1, 256);
    KR_INSTT(1, 2, 256); KR_INSTT(2, 2, 256); KR_INSTT(3, 2, 256); KR_INSTT(4, 2, 256); KR_INSTT(6, 2, 256); KR_INSTT(8, 2, 256);
    // several ranks emulated by one launch (krotov_group_iterate)
    KR_INSTTE(3, 0, 512); KR_INSTTE(3, 1, 256); KR_INSTTE(3, 2, 256); KR_INSTTE(6, 2, 256); KR_INSTTE(6, 0, 512);
}
}  // namespace kr
