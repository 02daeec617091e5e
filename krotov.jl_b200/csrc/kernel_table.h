// Table of the persistent warp-kernel instances.  The instances themselves are compiled in warp_inst_*.cu (one
// translation unit per family, so that the library builds in parallel); krotov_cuda.cu only looks them up.
#pragma once
#include <map>

#include "warp_kernel.cuh"

namespace kr {

using WarpKernel = void (*)(const WarpParams);
struct KernelKey {
    int W, LT, LPT = 32;
    bool operator<(const KernelKey &o) const {
        return W != o.W ? W < o.W : (LT != o.LT ? LT < o.LT : LPT < o.LPT);
    }
};
using KernelMap = std::map<KernelKey, WarpKernel>;

void add_warp_instances_runtime(KernelMap &t);  // runtime L, rows reloaded per use, up to 15 trajectory warps per CTA
void add_warp_instances_preg1(KernelMap &t);    // register-resident term rows, L = 1 and L = 3
void add_warp_instances_preg2(KernelMap &t);    // register-resident term rows, L = 2
void add_warp_instances_wide64(KernelMap &t);   // 64 threads (rows) per trajectory, 32 < d <= 64
void add_warp_instances_wide128(KernelMap &t);  // 128 threads per trajectory, 64 < d <= 128
void add_warp_instances_emul(KernelMap &t);     // several ranks emulated by one launch (krotov_group_iterate)
void add_warp2_instances(KernelMap &t);         // pair kernel: two trajectories of one generator per warp
void add_warp_instances_rf(KernelMap &t);       // replicated forward sweep of several ranks (one trajectory per warp, d <= 32)
void add_warp_instances_rf2(KernelMap &t);      // ... one / three controls, runtime L
void add_warp_instances_rf_emul(KernelMap &t);  // the same with the ranks emulated by one launch
// truncated-Taylor propagator (prop_method=Expmv), one warp per trajectory: the regular instances into `t`, the
// emulated-ranks instances into `emul` (maps of their own: the Chebyshev lookups above never see them)
void add_warp_instances_taylor(KernelMap &t, KernelMap &emul);

#define KR_INST(W, LT, MT) t[KernelKey{W, LT, 32}] = (WarpKernel)krotov_warp_kernel<W, LT, MT>
#define KR_INSTW(W, LT, MT, LPT) t[KernelKey{W, LT, LPT}] = (WarpKernel)krotov_warp_kernel<W, LT, MT, LPT>
#define KR_INSTE(W, LT, MT) t[KernelKey{W, LT, 32}] = (WarpKernel)krotov_warp_kernel<W, LT, MT, 32, true>
#define KR_INSTR(W, LT, MT) t[KernelKey{W, LT, 32}] = (WarpKernel)krotov_warp_kernel<W, LT, MT, 32, false, true>
#define KR_INSTRE(W, LT, MT) t[KernelKey{W, LT, 32}] = (WarpKernel)krotov_warp_kernel<W, LT, MT, 32, true, true>
#define KR_INSTT(W, LT, MT) t[KernelKey{W, LT, 32}] = (WarpKernel)krotov_warp_kernel<W, LT, MT, 32, false, false, true>
#define KR_INSTTE(W, LT, MT) emul[KernelKey{W, LT, 32}] = (WarpKernel)krotov_warp_kernel<W, LT, MT, 32, true, false, true>
#define KR_INST2(W, LT) t[KernelKey{W, LT, 32}] = (WarpKernel)krotov_warp2_kernel<W, LT>

}  // namespace kr
