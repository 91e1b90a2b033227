// backward stage-A edge kernel — instantiations + host dispatch
#include "pcd_kernels.h"
#include "pcd_launch.cuh"

namespace pcd {

template <int C, int S> struct KBwdA {
    static constexpr int kMinBlocks = 2; static const char* name() {
        return S == 1 ? (C == 4 ? "bwdA_c4_s1" : C == 8 ? "bwdA_c8_s1" : "bwdA_c16_s1")
                      : (C == 4 ? "bwdA_c4_s2" : C == 8 ? "bwdA_c8_s2" : "bwdA_c16_s2");
    }
    static PCD_D void run(const EdgeBwdArgs& a, int x, int y, int z, float* sm) { bwdA_body<C, S>(a, x, y, z, sm); }
};

#define GO_A(C_, S_) \
    return launch<KBwdA<C_, S_>, EdgeBwdArgs>(a, gx, gy, gz, bwdA_smem_floats(C_, S_, a.TH, a.TW, a.need_wgrad), stream)
int launch_bwdA(const EdgeBwdArgs& a, int c, int gx, int gy, int gz, void* stream) {
    if (a.S == 1) {
        if (c == 4) GO_A(4, 1); if (c == 8) GO_A(8, 1); if (c == 16) GO_A(16, 1);
    } else {
        if (c == 4) GO_A(4, 2); if (c == 8) GO_A(8, 2); if (c == 16) GO_A(16, 2);
    }
    return PCD_ERR_UNSUPPORTED;
}

}  // namespace pcd
