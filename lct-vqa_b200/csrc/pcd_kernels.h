// pcd_kernels.h — host launchers of the edge kernels; each lives in its own translation unit so the
// heavy template instantiations compile in parallel.
#pragma once
#include "pcd_edge.cuh"

namespace pcd {
// generic edge kernels (pcd_edge.cuh): any geometry, run-time tile a.TH x a.TW
int launch_fwdA(const PassArgs& a, int c, int gx, int gy, int gz, void* stream);
int launch_fwdB(const PassArgs& a, int c, int gx, int gy, int gz, void* stream);
int launch_bwdA(const EdgeBwdArgs& a, int c, int gx, int gy, int gz, void* stream);
int launch_bwdB(const EdgeBwdArgs& a, int c, int gx, int gy, int gz, void* stream);
// stage-B data and weight-gradient backward (pcd_edge_bwd2.cuh): production geometries only; a.TH / a.TW hold the tile (TW == Wo)
bool bwd2_tile(int c, int S, int Ho, int Wo, int* TH);
int launch_bwdB2(const EdgeBwdArgs& a, int c, int gz, void* stream);
int launch_wgrad2(const EdgeBwdArgs& a, int c, int gz, void* stream);
// v4 forward (pcd_edge_v4.cuh): stage A + stage B of a group of production-geometry edges
struct FwdV4Args;
bool fwd4_supported(int c, int S, int Ho, int Wo);
int launch_fwd4(const FwdV4Args& a, int c, int S, void* stream);
// v4 stage-A backward data kernels (pcd_edge_bwd4.cuh): plain stores into the two partial-grad slots of every edge
int launch_bwdA4(const EdgeBwdArgs& a, int c, int nedges, void* stream);
struct PreArgs;
struct PreBwdArgs;
int launch_pre_conv(const PreArgs& a, void* stream);
// tensor-core (tcgen05) preprocess kernels, pcd_pre_tc.cu: plain 1x1 ReLUConvBN at the production shapes
bool pre_tc_supported(int B, int Cin, int Cout, int H, int W, int fr);
int launch_pre_tc_fwd(const PreArgs& a, void* stream);
int launch_pre_tc_bwd(const PreBwdArgs& a, void* stream);
int launch_pre_bwd(const PreBwdArgs& a, void* stream);
// stand-alone candidate operations on all channels (pcd_opk.cuh): the derived-architecture network's ops
struct DwArgs;
struct PwArgs;
struct PoolArgs;
struct AffineArgs;
int launch_dw_fwd(const DwArgs& a, int KS, void* stream);
int launch_dw_bwd(const DwArgs& a, int KS, void* stream);
int launch_pw_fwd(const PwArgs& a, void* stream);
int launch_pw_bwd(const PwArgs& a, void* stream);
int launch_pool_fwd(const PoolArgs& a, void* stream);
int launch_pool_bwd(const PoolArgs& a, void* stream);
int launch_affine(const AffineArgs& a, void* stream);
}  // namespace pcd
