"""Build recipes for the native library (in-tree, so the .so travels with the repo snapshot).

    build_cuda()  -> lct-vqa_b200/libpcdarts_sm100.so   nvcc, sm_100a only (cross-compiles without a GPU)
    build_emu()   -> tests/emu/libpcd_emu.so            g++ -DPCD_EMU: CPU emulation of the same kernel
                                                         sources, TEST INFRASTRUCTURE ONLY
"""
import os
import shutil
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
SOURCES = [os.path.join(CSRC, f) for f in ("pcd_api.cu", "pcd_k_fwd.cu", "pcd_k_fwd4.cu", "pcd_k_bwd4.cu", "pcd_k_bwdA.cu", "pcd_k_bwdB.cu", "pcd_k_bwd2.cu", "pcd_k_pre.cu", "pcd_pre_tc.cu", "pcd_gemm_sm100.cu", "pcd_ce.cu", "pcd_lstm.cu", "pcd_decode.cu", "pcd_flat.cu", "pcd_gemm_small.cu", "pcd_k_ops.cu", "pcd_k_eval.cu", "pcd_droppath.cu")]
HEADERS = [os.path.join(CSRC, f) for f in ("pcd_common.cuh", "pcd_edge.cuh", "pcd_fwd.cuh", "pcd_bwd.cuh",
                                           "pcd_launch.cuh", "pcd_kernels.h", "pcd_pre.cuh", "pcd_edge_bwd2.cuh", "pcd_edge_v4.cuh", "pcd_edge_bwd4.cuh", "pcd_tc.cuh", "pcd_opk.cuh", "pcd_eval.cuh", "pcd_philox.cuh")] + \
          [os.path.join(ROOT, "include", "pcdarts_sm100.h")]
BUILD_DIR = os.path.join(HERE, "build")
CUDA_LIB = os.path.join(HERE, "libpcdarts_sm100.so")
EMU_LIB = os.path.join(ROOT, "tests", "emu", "libpcd_emu.so")

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "--expt-relaxed-constexpr", "--expt-extended-lambda", "-Xcompiler", "-fPIC"]


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def nvcc_path():
    return shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"


def _compile_all(cmd_for, objs_dir, verbose=False):
    """Compile every source to an object file, all translation units in parallel."""
    os.makedirs(objs_dir, exist_ok=True)
    procs, objs = [], []
    for src in SOURCES:
        obj = os.path.join(objs_dir, os.path.basename(src) + ".o")
        objs.append(obj)
        procs.append((src, subprocess.Popen(cmd_for(src, obj), stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    log = ""
    for src, p in procs:
        out, _ = p.communicate()
        log += out
        if p.returncode != 0:
            for _, q in procs:
                if q.poll() is None:
                    q.kill()
            raise RuntimeError(f"compiling {src} failed:\n{out}")
    if verbose:
        print(log)
    return objs


def build_cuda(force=False, verbose=False):
    if not force and not _stale(CUDA_LIB, SOURCES + HEADERS):
        return CUDA_LIB
    nvcc = nvcc_path()
    extra = ["-Xptxas", "-v"] if verbose else []
    objs = _compile_all(lambda src, obj: [nvcc] + NVCC_FLAGS + extra + ["-c", "-o", obj, src],
                        os.path.join(BUILD_DIR, "cuda"), verbose)
    r = subprocess.run([nvcc, "-shared", "-o", CUDA_LIB] + objs, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc link failed:\n" + r.stdout + r.stderr)
    return CUDA_LIB


def build_emu(force=False):
    if not force and not _stale(EMU_LIB, SOURCES + HEADERS):
        return EMU_LIB
    os.makedirs(os.path.dirname(EMU_LIB), exist_ok=True)
    objs = _compile_all(lambda src, obj: ["g++", "-O2", "-std=c++17", "-DPCD_EMU", "-x", "c++", "-fPIC", "-c", "-o", obj, src],
                        os.path.join(BUILD_DIR, "emu"))
    r = subprocess.run(["g++", "-shared", "-o", EMU_LIB] + objs, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("g++ (emulation build) link failed:\n" + r.stdout + r.stderr)
    return EMU_LIB
