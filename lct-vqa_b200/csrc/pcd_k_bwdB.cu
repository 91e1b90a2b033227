// backward stage-B edge kernel — instantiations + host dispatch
#include "pcd_kernels.h"
#include "pcd_launch.cuh"

namespace pcd {

template <int C> struct KBwdB {
    static constexpr int kMinBlocks = 2; static const char* name() { return C == 4 ? "bwdB_c4" : C == 8 ? "bwdB_c8" : "bwdB_c16"; }
    static PCD_D void run(const EdgeBwdArgs& a, int x, int y, int z, float* sm) { bwdB_body<C>(a, x, y, z, sm); }
};

#define GO_B(C_) \
    return launch<KBwdB<C_>, EdgeBwdArgs>(a, gx, gy, gz, bwdB_smem_floats(C_, a.TH, a.TW, a.need_wgrad), stream)
int launch_bwdB(const EdgeBwdArgs& a, int c, int gx, int gy, int gz, void* stream) {
    if (c == 4) GO_B(4); if (c == 8) GO_B(8); if (c == 16) GO_B(16);
    return PCD_ERR_UNSUPPORTED;
}

}  // namespace pcd
