// eval-mode kernels (pcd_eval.cuh) — instantiations + host launchers
#include "pcd_eval.cuh"
#include "pcd_launch.cuh"

namespace pcd {

template <int C> struct KEvalNode {
    static constexpr int kMinBlocks = 2;
    static const char* name() { return C == 4 ? "eval_node_c4" : C == 8 ? "eval_node_c8" : "eval_node_c16"; }
    static PCD_D void run(const EvalNodeArgs& a, int x, int y, int, float* sm) { eval_node_body<C>(a, x, y, sm); }
};
struct KEvalPre {
    static constexpr int kMinBlocks = 2;
    static const char* name() { return "eval_pre"; }
    static PCD_D void run(const EvalPreArgs& a, int x, int y, int z, float* sm) { eval_pre_body(a, x, y, z, sm); }
};
struct KEvalStem {
    static constexpr int kMinBlocks = 2;
    static const char* name() { return "eval_stem"; }
    static PCD_D void run(const EvalStemArgs& a, int x, int y, int, float* sm) { eval_stem_body(a, x, y, sm); }
};

int launch_eval_node(const EvalNodeArgs& a, int c, void* stream) {
    const int tiles = (a.Ho + a.TH - 1) / a.TH;
    const size_t sm = eval_smem(c, a.TH, a.Wo, a.maxS).total;
    if (c == 4) return launch<KEvalNode<4>, EvalNodeArgs>(a, tiles, a.B, 1, sm, stream);
    if (c == 8) return launch<KEvalNode<8>, EvalNodeArgs>(a, tiles, a.B, 1, sm, stream);
    if (c == 16) return launch<KEvalNode<16>, EvalNodeArgs>(a, tiles, a.B, 1, sm, stream);
    return PCD_ERR_UNSUPPORTED;
}

int launch_eval_pre(const EvalPreArgs& a, void* stream) {
    if (a.Cout % kEvalPreCO || (a.fr && (a.Cout / 2) % kEvalPreCO)) return PCD_ERR_UNSUPPORTED;
    const int gx = (a.Ho * a.Wo + kEvalPrePx - 1) / kEvalPrePx;
    return launch<KEvalPre, EvalPreArgs>(a, gx, a.B, a.Cout / kEvalPreCO, eval_pre_smem_floats(), stream);
}

int launch_eval_stem(const EvalStemArgs& a, void* stream) {
    const int gx = (a.H + a.rows - 1) / a.rows;
    return launch<KEvalStem, EvalStemArgs>(a, gx, a.B, 1, eval_stem_smem_floats(a.Cout, a.rows, a.W), stream);
}

}  // namespace pcd
