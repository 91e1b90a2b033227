// production backward edge kernels (pcd_edge_bwd2.cuh: stage-B data, weight gradients) — instantiations + host dispatch
#include "pcd_edge_bwd2.cuh"
#include "pcd_kernels.h"
#include "pcd_launch.cuh"

namespace pcd {

template <int C, int TH, int TW> struct KBwdB2 {
    static constexpr int kMinBlocks = 4;      // 64 registers, 44-52 KB
    static const char* name() { return C == 4 ? "bwdB_c4" : C == 8 ? "bwdB_c8" : "bwdB_c16"; }
    static PCD_D void run(const EdgeBwdArgs& a, int x, int y, int z, float* sm) { bwdB2_body<C, TH, TW>(a, x, y, z, sm); }
};
template <int C, int S, int TH, int TW> struct KWgrad2 {
    static constexpr int kMinBlocks = 2;
    static const char* name() {
        return S == 1 ? (C == 4 ? "wgrad_c4_s1" : C == 8 ? "wgrad_c8_s1" : "wgrad_c16_s1") : (C == 8 ? "wgrad_c8_s2" : "wgrad_c16_s2");
    }
    static PCD_D void run(const EdgeBwdArgs& a, int x, int y, int z, float* sm) { wgrad2_body<C, S, TH, TW>(a, x, y, z, sm); }
};

// tiles: full output width, TH rows; these kernels exist for the five production edge geometries
bool bwd2_tile(int c, int S, int Ho, int Wo, int* TH) {
    int th = 0;
    if (S == 1) {
        if (c == 4 && Wo == 64) th = 16;
        else if (c == 8 && Wo == 32) th = 16;
        else if (c == 16 && Wo == 16) th = 16;
    } else {
        if (c == 8 && Wo == 32) th = 8;
        else if (c == 16 && Wo == 16) th = 8;
    }
    if (!th || Ho % th) return false;
    *TH = th;
    return true;
}

template <class K>
static int go2(const EdgeBwdArgs& a, int gz, size_t smem_floats, void* stream) {
    return launch<K, EdgeBwdArgs>(a, a.Ho / a.TH, a.B, gz, smem_floats, stream);
}
int launch_bwdB2(const EdgeBwdArgs& a, int c, int gz, void* stream) {
    if (c == 4 && a.TH == 16 && a.TW == 64) return go2<KBwdB2<4, 16, 64>>(a, gz, bwdB2_smem_floats<4, 16, 64>(), stream);
    if (c == 8 && a.TH == 16 && a.TW == 32) return go2<KBwdB2<8, 16, 32>>(a, gz, bwdB2_smem_floats<8, 16, 32>(), stream);
    if (c == 16 && a.TH == 16 && a.TW == 16) return go2<KBwdB2<16, 16, 16>>(a, gz, bwdB2_smem_floats<16, 16, 16>(), stream);
    return PCD_ERR_UNSUPPORTED;
}
template <class K>
static int go_w(const EdgeBwdArgs& a, int gz, size_t smem_floats, void* stream) {
    return launch<K, EdgeBwdArgs>(a, 1, (a.B + kWgradImages - 1) / kWgradImages, gz, smem_floats, stream);
}
int launch_wgrad2(const EdgeBwdArgs& a, int c, int gz, void* stream) {
    if (a.S == 1) {
        if (c == 4 && a.TH == 16 && a.TW == 64) return go_w<KWgrad2<4, 1, 16, 64>>(a, gz, wgrad2_smem_floats<4, 1, 16, 64>(), stream);
        if (c == 8 && a.TH == 16 && a.TW == 32) return go_w<KWgrad2<8, 1, 16, 32>>(a, gz, wgrad2_smem_floats<8, 1, 16, 32>(), stream);
        if (c == 16 && a.TH == 16 && a.TW == 16) return go_w<KWgrad2<16, 1, 16, 16>>(a, gz, wgrad2_smem_floats<16, 1, 16, 16>(), stream);
    } else {
        if (c == 8 && a.TH == 8 && a.TW == 32) return go_w<KWgrad2<8, 2, 8, 32>>(a, gz, wgrad2_smem_floats<8, 2, 8, 32>(), stream);
        if (c == 16 && a.TH == 8 && a.TW == 16) return go_w<KWgrad2<16, 2, 8, 16>>(a, gz, wgrad2_smem_floats<16, 2, 8, 16>(), stream);
    }
    return PCD_ERR_UNSUPPORTED;
}

}  // namespace pcd
