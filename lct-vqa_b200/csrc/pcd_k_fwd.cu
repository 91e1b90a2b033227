// forward edge kernels (stage A / stage B) — instantiations + host dispatch
#include "pcd_kernels.h"
#include "pcd_launch.cuh"

namespace pcd {

template <int C, int S> struct KFwdA {
    static constexpr int kMinBlocks = 3; static const char* name() {
        return S == 1 ? (C == 4 ? "fwdA_c4_s1" : C == 8 ? "fwdA_c8_s1" : "fwdA_c16_s1")
                      : (C == 4 ? "fwdA_c4_s2" : C == 8 ? "fwdA_c8_s2" : "fwdA_c16_s2");
    }
    static PCD_D void run(const PassArgs& a, int x, int y, int z, float* sm) { fwdA_body<C, S>(a, x, y, z, sm); }
};
template <int C> struct KFwdB {
    static constexpr int kMinBlocks = 3; static const char* name() { return C == 4 ? "fwdB_c4" : C == 8 ? "fwdB_c8" : "fwdB_c16"; }
    static PCD_D void run(const PassArgs& a, int x, int y, int z, float* sm) { fwdB_body<C>(a, x, y, z, sm); }
};

#define GO_A(C_, S_) return launch<KFwdA<C_, S_>, PassArgs>(a, gx, gy, gz, fwdA_smem_floats(C_, S_, a.TH, a.TW), stream)
int launch_fwdA(const PassArgs& a, int c, int gx, int gy, int gz, void* stream) {
    if (a.S == 1) {
        if (c == 4) GO_A(4, 1); if (c == 8) GO_A(8, 1); if (c == 16) GO_A(16, 1);
    } else {
        if (c == 4) GO_A(4, 2); if (c == 8) GO_A(8, 2); if (c == 16) GO_A(16, 2);
    }
    return PCD_ERR_UNSUPPORTED;
}

#define GO_B(C_) return launch<KFwdB<C_>, PassArgs>(a, gx, gy, gz, fwdB_smem_floats(C_, a.TH, a.TW), stream)
int launch_fwdB(const PassArgs& a, int c, int gx, int gy, int gz, void* stream) {
    if (c == 4) GO_B(4); if (c == 8) GO_B(8); if (c == 16) GO_B(16);
    return PCD_ERR_UNSUPPORTED;
}

}  // namespace pcd
