#!/usr/bin/env python
"""bench.py — search steps/sec of the PC-DARTS-VQA search step on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo (sm_100a kernels)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path (oracle port), rank 0 only

One "step" = the alpha-step (unrolled, finite-difference Hessian-vector product; --first-order for the
first-order architect) followed by the w-step of darts_vqa/experiment.py:176-200 on one synthetic batch
of B=64 per GPU (64x64 images, 30-token questions, V=17858, 1000 answers, C=16, 4 cells).  For N>1 the
driver launches one rank per GPU with torchrun; the batch is sharded (weak scaling: 64 per GPU) and
gradients are averaged with NCCL.

Prints ONE JSON line (rank 0).  value = whole-job 64-sample search steps per second with inputs
resident in HBM; e2e = the same through the public API with host (pinned) inputs copied inside the
timed region and the loss read back; roofline = MixedOp kernel group measured with per-launch CUDA
events in a separate profiled region; cpu_baseline = the oracle port on the host cores (bounded sample).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "lct-vqa_b200")
for p in (PKG, ROOT):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

_REAL_STDOUT = 1
METRIC = "search steps/sec (w+alpha step)"
UNIT = "steps/s"
DIMS = dict(embed_size=512, ans_vocab_size=1000, word_embed_size=300, num_layers=1, hidden_size=512)
# SURVEY.md §8(d): algorithmic bytes of all 56 MixedOp edges at B=64 (fwd 1241.5 MB, fwd+bwd 2977.5 MB)
MIXED_FWD_MB_B64, MIXED_BWD_MB_B64 = 1241.5136, 1736.0
MIXED_KERNELS = ("fwdA", "fwdB", "combine", "node_stats", "bwdB", "bwdA", "wgrad", "SourceGrad", "ArchGrads")
EDGE_SHAPES = [("T1 C16@64 s1", 16, 1, 64, 14), ("T2 C32 64->32 s2", 32, 2, 64, 8), ("T3 C32@32 s1", 32, 1, 32, 6),
               ("T4 C64 32->16 s2", 64, 2, 32, 8), ("T5 C64@16 s1", 64, 1, 16, 20)]


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=64, help="per-GPU batch (reference default 64)")
    ap.add_argument("--vocab", type=int, default=17858)
    ap.add_argument("--img", type=int, default=64)
    ap.add_argument("--first-order", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="do not capture the step in a CUDA graph")
    ap.add_argument("--no-graph-dp", action="store_true", help="under data parallelism run the step eagerly instead of as a CUDA graph with the NCCL all-reduces captured inside")
    ap.add_argument("--no-parity", action="store_true", help="N>1: skip the replica-checksum / averaged-gradient-vs-oracle block")
    ap.add_argument("--concurrent-hvp", action="store_true", help="run the two finite-difference passes of the Hessian-vector product as two graph branches (model | twin); measured 2 % slower than one after the other on B200, so off by default")
    ap.add_argument("--no-overlap", action="store_true", help="keep the weight-grad jobs on the main stream")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed (loss, "
                    "alphas / betas, BatchNorm running statistics, a fixed sample of the weights) as DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs applies to --impl b200 only: the reference arm's CPU path is not the timed GPU path")
    return a


def workload(a, n):
    return {"workload": f"PC-DARTS-VQA search step: {'first-order' if a.first_order else 'unrolled (HVP)'} alpha-step"
                        f" + w-step, VqaModel(512,{a.vocab},1000,300,1,512,'darts'), C=16, 4 cells, {a.img}x{a.img}",
            "batch_per_gpu": a.batch, "global_batch": a.batch * n, "parallelism": f"dp{n}", "unrolled": not a.first_order,
            "l2": "no flush needed: each pass streams ~1.8 GB of saved activations at B=64 (>> 126 MB L2); "
                  "the MixedOp micro-benchmark flushes L2 with a 512 MB write between iterations"}


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def step_traffic(unrolled, batch):
    """DRAM bytes per step of the MixedOp kernel group: dram__bytes_read.sum + dram__bytes_write.sum summed over the group's
    launches in the committed whole-step ncu launch list (profiles/tools/launch_traffic.py writes the JSON from the csv).
    None when the list for the current kernels is absent — never a stale constant."""
    path = os.path.join(ROOT, "profiles", "r02_step_traffic.json")
    try:
        with open(path) as f:
            t = json.load(f)
        key = "unrolled" if unrolled else "first_order"
        return t[key]["mixedop_group_bytes"] * batch / t["batch"], \
            f"ncu cold-cache DRAM counters over one whole step at B={t['batch']} ({t['source']}), scaled by B/{t['batch']}"
    except Exception:
        return None, "no ncu launch list for the current kernels under profiles/"


def synth_batch(seed, B, V, img):
    g = torch.Generator().manual_seed(seed)
    image = torch.randn(B, 3, img, img, generator=g)
    qst = torch.randint(0, V, (B, 30), generator=g)
    qst[:, 0] = 2
    lbl = torch.randint(0, 1000, (B,), generator=g)
    return image, qst, lbl


DUMP_WEIGHT_SAMPLE = 1 << 22        # 16 MB of float32; all weights are ~95 MB at V = 17858


def dump_outputs(path, model, loss):
    """What the timed step hands its caller, as float32 .npy files under `path`: the loss of the last step and the state
    that step left behind (alphas / betas, BatchNorm running statistics, weights).  The weights are a sample: positions drawn
    with a fixed seed from all parameters concatenated in model.parameters() order, so equal shapes give equal positions.
    The inputs are seeded, but the kernels reduce BatchNorm sums and split-K products with atomics: two runs of one build
    agree to that rounding as it grows over the steps, not bit for bit."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    with torch.no_grad():
        out = {"loss": loss.reshape(1)}
        out.update(zip(("alphas_normal", "alphas_reduce", "betas_normal", "betas_reduce"), model.arch_parameters()))
        out["bn_running_stats"] = torch.cat([b.reshape(-1) for b in model.buffers() if b.is_floating_point()])
        flat = torch.cat([p.reshape(-1) for p in model.parameters()])
        idx = torch.randperm(flat.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_WEIGHT_SAMPLE].sort().values
        out["weights_sample"] = flat[idx.to(flat.device)]
        for name, t in out.items():
            np.save(os.path.join(path, name + ".npy"), t.detach().float().cpu().numpy())


# ------------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle port of the reference's CPU path (oracle/pcdarts_oracle.py)
# ------------------------------------------------------------------------------------------------------
def cpu_search_step_factory(a, B):
    from oracle import pcdarts_oracle as O
    torch.manual_seed(10)
    sd = O.alloc_state(O.vqa_spec(qst_vocab_size=a.vocab, **DIMS), seed=10)
    par, buf = O.split_state(sd)
    for v in par.values():
        v.requires_grad_(True)
    arch = [(1e-3 * torch.randn(s)).requires_grad_(True) for s in ((14, 8), (14, 8), (14,), (14,))]
    keys = list(par.keys())
    train, valid = synth_batch(10, B, a.vocab, a.img), synth_batch(11, B, a.vocab, a.img)
    st_a, st_w, bns = {}, {}, O.BNState(buf)

    def step():
        O.architect_step(par, bns, arch, st_a, train, valid, 1e-3, keys, unrolled=not a.first_order)
        return float(O.w_step(par, bns, arch, train, st_w, keys))
    return step


def time_cpu(a, steps, warmup, budget_s):
    """Time the oracle port of the reference's CPU path on the FULL per-GPU batch, all host cores.

    The sample is bounded by timing fewer steps, never fewer samples (cost is not linear in the batch on a CPU): at most
    `steps` steps, stopping early once the next one would overrun `budget_s`; at least one.  The same function serves the
    `cpu_baseline` of the GPU arm (steps=1) and `--impl reference`, so the two numbers of one record agree.  Only when a
    single full-batch step cannot fit the budget at all is the batch halved (and the scaling stated)."""
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    t0 = time.time()
    probe = cpu_search_step_factory(a, min(2, a.batch))
    probe()                                  # allocator / thread-pool / dispatch warm-up (2 samples, untimed)
    t1 = time.time()
    probe()
    per_sample = (time.time() - t1) / min(2, a.batch)
    B = a.batch
    while B > 2 and per_sample * B * 0.5 > budget_s:       # 0.5: measured, large batches amortise per-op overheads
        B //= 2
    step = cpu_search_step_factory(a, B)
    t_begin = time.time()
    done_w = 0
    if warmup > 0 and per_sample * B * 0.5 * 3 <= budget_s:   # one full-size warm-up step when three steps fit
        step()
        done_w = 1
    times = []
    for _ in range(max(1, steps)):
        if times and (time.time() - t_begin) + sum(times) / len(times) > budget_s:
            break
        t = time.time()
        step()
        times.append(time.time() - t)
    dt = sum(times) / len(times)
    value = (1.0 / dt) * (B / a.batch)
    note = "" if B == a.batch else f"; ONE full-batch step exceeds the {budget_s:.0f} s budget on this host, value scaled by {B}/{a.batch}"
    return value, dt, {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "steps_timed": len(times),
                       "samples_per_step": B,
                       "sample": f"{len(times)} timed step(s) (+{done_w} full-size warm-up) of the same search step on {B} of the "
                                 f"{a.batch} samples of the batch, {dt:.2f} s each, {cores} threads{note}; model setup and a "
                                 f"2-sample warm-up ({t_begin - t0:.1f} s) not timed"}


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    value, dt, cb = time_cpu(a, a.steps, a.warmup, budget_s=150.0)
    emit({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
        "steps_timed": cb["steps_timed"], "warmup": a.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": workload(a, a.gpus), "cpu_baseline": cb,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0})


# ------------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.lines, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line)

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for line in self.lines:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx = float(f[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------
# this repo's arm
# ------------------------------------------------------------------------------------------------------
def run_b200(a):
    import torch.distributed as dist
    import config
    import pcd_dist as pdist
    import pcd_native
    from argparse import Namespace

    rank, world = pdist.init_from_env()
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    config.DEVICE = dev
    lib = pcd_native.load_cuda()
    import pcd_ops
    pcd_ops.set_wgrad_overlap(not a.no_overlap)      # weight-grad jobs on the library's low-priority stream
    from pcdarts.architect_vqa import Architect
    from search import SearchStep
    from vqa_model import VqaModel

    torch.manual_seed(10)
    model = VqaModel(qst_vocab_size=a.vocab, img_encoder_type="darts", **DIMS).to(dev).train()
    reducer = pdist.GradReducer() if world > 1 else None
    if world > 1:           # identical replicas: rank 0's init everywhere
        for t in list(model.parameters()) + list(model.buffers()) + list(model.arch_parameters()):
            dist.broadcast(t.data, 0)
    use_graph = not a.no_graph and (world == 1 or not a.no_graph_dp)
    import pcd_flat
    opt = pcd_flat.FlatAdam(model.parameters(), lr=1e-3)       # torch.optim.Adam's update, one launch over the flat runs
    architect = Architect(model, Namespace(arch_learn_rate=6e-4, arch_wt_decay=1e-3, qst_only=False), reducer=reducer)
    if use_graph:
        architect.optimizer = torch.optim.Adam(model.arch_parameters(), lr=6e-4, betas=(0.5, 0.999), weight_decay=1e-3,
                                               capturable=True)
    architect.concurrent_hvp = bool(a.concurrent_hvp)      # w + R v on the model | w - R v on the twin: two graph branches
    stepper = SearchStep(model, architect, opt, reducer=reducer)
    host_train = [t.pin_memory() for t in synth_batch(10 + rank, a.batch, a.vocab, a.img)]
    host_valid = [t.pin_memory() for t in synth_batch(1010 + rank, a.batch, a.vocab, a.img)]
    train = [t.to(dev) for t in host_train]
    valid = [t.to(dev) for t in host_valid]
    unrolled = not a.first_order

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            dist.barrier()
        return ms.item()

    graphed = None
    if use_graph:
        from search import GraphedSearchStep
        graphed = GraphedSearchStep(stepper, train, valid, 1e-3, unrolled=unrolled)

    last_loss = [None]

    def step_resident():
        if graphed is not None:
            last_loss[0] = graphed()
        else:
            last_loss[0] = stepper.step(train, valid, 1e-3, unrolled=unrolled)

    def step_e2e():
        if graphed is not None:
            return graphed(host_train, host_valid).item()      # pinned host -> static device buffers, replay, read loss
        tr = [t.to(dev, non_blocking=True) for t in host_train]
        va = [t.to(dev, non_blocking=True) for t in host_valid]
        return stepper.step(tr, va, 1e-3, unrolled=unrolled).item()

    for _ in range(max(a.warmup, 3)):
        step_resident()
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    l0 = lib.pcd_launch_count()
    ms = timed(step_resident, a.steps)
    launches = lib.pcd_launch_count() - l0
    clk = clocks.stop() if rank == 0 else None      # the clock record covers the timed steps only
    if a.dump_outputs and rank == 0:        # before anything below steps the model again
        dump_outputs(a.dump_outputs, model, last_loss[0])
    if graphed is not None:      # replays do not pass through the host launcher: count one eager step instead
        l0 = lib.pcd_launch_count()
        stepper.step(train, valid, 1e-3, unrolled=unrolled)
        launches = (lib.pcd_launch_count() - l0) * a.steps
    value = world * a.steps / (ms / 1e3)

    step_e2e()
    ms_e2e = timed(step_e2e, a.steps)
    h2d = 2 * sum(t.numel() * t.element_size() for t in host_train)
    e2e = {"value": world * a.steps / (ms_e2e / 1e3), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
           "ms_per_step": ms_e2e / a.steps}

    # ---- per-launch CUDA-event profile of this library's kernels (separate region: events perturb) ----
    hbm, peak_src = peaks()
    roofline, by_kernel = None, {}
    nprof = 2
    pcd_ops.set_wgrad_overlap(False)       # per-kernel event times are only meaningful without concurrent kernels
    lib.pcd_profile_enable(1)              # every rank runs the same steps (they contain collectives)
    for _ in range(nprof):
        stepper.step(train, valid, 1e-3, unrolled=unrolled)      # eager: the event profiler lives in the host launcher
    torch.cuda.synchronize()
    prof = pcd_native.profile_collect(lib)
    lib.pcd_profile_enable(0)
    pcd_ops.set_wgrad_overlap(not a.no_overlap)
    if rank == 0:
        total_ms = sum(v[0] for v in prof.values())
        for k, (t, c) in sorted(prof.items(), key=lambda kv: -kv[1][0]):
            by_kernel[k] = {"ms_per_step": t / nprof, "launches_per_step": c / nprof, "share": t / total_ms}
        mixed_ms = sum(t for k, (t, c) in prof.items() if k.startswith(MIXED_KERNELS)) / nprof
        n_fwd = 5 if unrolled else 2
        n_bwd = 5 if unrolled else 2
        alg_mb = (n_fwd * MIXED_FWD_MB_B64 + n_bwd * MIXED_BWD_MB_B64) * a.batch / 64.0
        achieved = alg_mb / 1e3 / (mixed_ms / 1e3)
        fam = {}
        for k, (t, c) in prof.items():       # kernel families: template / geometry suffixes (_c4, _s1, ...) folded together
            if k.startswith(MIXED_KERNELS):
                f = next(m for m in MIXED_KERNELS if k.startswith(m))
                fam[f] = fam.get(f, 0.0) + t / nprof
        top = max(fam, key=fam.get) if fam else next(iter(by_kernel))
        traffic, traffic_note = step_traffic(unrolled, a.batch)
        roofline = {"bound": "hbm", "kernel": "MixedOp kernel group (fwdA,fwdB,combine | node_stats,bwdB,bwdA,wgrad,"
                                              "source_grad,arch_grads): all 56 edges x all passes of one step",
                    "achieved": achieved, "peak": hbm, "unit": "GB/s", "frac": achieved / hbm,
                    "traffic": traffic, "traffic_note": traffic_note, "ms_by_family": fam,
                    "algorithmic_mb_per_step": alg_mb, "kernel_ms_per_step": mixed_ms, "peak_source": peak_src,
                    "passes_per_step": {"forward": n_fwd, "backward": n_bwd},
                    "dominant_kernel": top, "native_kernel_ms_per_step": total_ms / nprof,
                    "share_of_step": (total_ms / nprof) / (ms / a.steps), "by_kernel": by_kernel}

    extras = {}
    roofline_gemm = None
    if rank == 0 and not a.no_extras:
        try:
            roofline_gemm = gemm_roofline(a, dev)
        except Exception as e:
            roofline_gemm = {"error": repr(e)[:200]}
    if not a.no_extras:
        if rank == 0:
            extras["mixedop_fwd_bwd"] = mixedop_microbench(dev, a.batch, hbm)
            # SURVEY.md §8(d): roofline sweep of a single MixedOp at larger per-GPU batches (one edge at B=64 is latency-bound)
            extras["mixedop_fwd_bwd_b256"] = mixedop_microbench(dev, 256, hbm)
            extras["mixedop_fwd_bwd_b512"] = mixedop_microbench(dev, 512, hbm)
        if True:
            w_ms = timed(lambda: stepper.w_step(*train), max(3, a.steps // 2)) / max(3, a.steps // 2)
            fo_ms = timed(lambda: stepper.step(train, valid, 1e-3, unrolled=False), max(3, a.steps // 2)) / max(3, a.steps // 2)
            extras["w_step_only_steps_per_s"] = world * 1e3 / w_ms
            extras["w_plus_first_order_alpha_steps_per_s"] = world * 1e3 / fo_ms
    if rank == 0 and world == 1 and not a.no_extras:
        # BASELINE.json configs[2]: the 3-stage LCT alpha-step (6 forward / 5 backward search-net passes + VGG19 W model), eager
        try:
            extras["lct_alpha_step"] = lct_alpha_step_bench(a, dev)
        except Exception as e:      # the headline numbers above do not depend on it
            extras["lct_alpha_step"] = {"error": repr(e)[:200]}
        try:
            extras["derived_network_train_pass"] = derived_network_bench(model, dev)
        except Exception as e:
            extras["derived_network_train_pass"] = {"error": repr(e)[:200]}
    parity = None
    if world > 1 and not a.no_parity:
        parity = dp_parity(a, model, reducer, rank, world, dev, stepper=stepper)
    cpu = None
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        _, _, cpu = time_cpu(a, 1, 0, budget_s=45.0)
    if rank == 0:
        out = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 3),
               "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
               "data": "synthetic", "config": workload(a, world), "e2e": e2e, "gpu_launches": int(launches), "cuda_graph": bool(use_graph),
               "wgrad_overlap": not a.no_overlap, "concurrent_hvp": bool(a.concurrent_hvp), "clocks": clk, "roofline": roofline, "roofline_gemm": roofline_gemm, "cpu_baseline": cpu, "extras": extras,
               "parity": parity,
               "comm": None if reducer is None else reducer.report()}
        emit(out)
    if world > 1:
        torch.cuda.synchronize()
        dist.barrier()
        if use_graph:
            # NCCL kernels live inside the captured graph: tearing the communicator down under it hung once
            # (profiles/r01_bench_dp2_graph.json run); every rank has reported, so leave without the teardown
            sys.stdout.flush()
            sys.stderr.flush()
            os._exit(0)
        dist.destroy_process_group()


def dp_parity(a, model, reducer, rank, world, dev, shard_batch=None, stepper=None):
    """NCCL parity evidence (VERDICT r01 weak #3), after the timed steps, on every rank (it contains collectives):
      1. replica consistency: per-rank fp64 checksums (sum, sum of squares, over every weight and alpha/beta) all-gathered;
         data-parallel replicas must stay BIT-identical;
      2. one w-step forward/backward on a fresh shard of `shard_batch` samples per rank (dropout off), gradients averaged by
         the GradReducer over NCCL, compared on rank 0 with the oracle's gradients of the same `world` shards averaged by hand
         (the only place this arm executes oracle/: as the checker)."""
    import torch.distributed as dist
    # the oracle's cost is bounded by the TOTAL number of samples (16, as 2 x 8 at N = 2), not by the rank count; the other ranks
    # wait on a gloo barrier (a blocking socket wait): an NCCL barrier spins one host core per rank and, with the oracle's
    # OpenMP threads oversubscribed, an 8-rank run took > 8 minutes here
    if shard_batch is None:
        shard_batch = max(2, 16 // world)
    cpu_group = None
    try:
        import datetime
        cpu_group = dist.new_group(backend="gloo", timeout=datetime.timedelta(seconds=120))
        ok = torch.ones(1, device=dev)
    except Exception:
        ok = torch.zeros(1, device=dev)
    dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    if float(ok) < 1.0:      # some rank has no gloo group: everybody falls back to the (spinning) NCCL barrier
        cpu_group = None
    with torch.no_grad():
        tensors = [p.detach() for p in model.parameters()] + [t.detach() for t in model.arch_parameters()]
        arch = [t.detach() for t in model.arch_parameters()]
        gn = getattr(getattr(stepper, "eager", stepper), "last_grad_norm", None) if stepper is not None else None
        cs = torch.stack([torch.stack([t.double().sum() for t in tensors]).sum(),
                          torch.stack([(t.double() ** 2).sum() for t in tensors]).sum(),
                          torch.stack([t.double().sum() for t in arch]).sum(),
                          (gn.detach().double().reshape(()) if torch.is_tensor(gn) else torch.zeros((), dtype=torch.float64, device=dev))])
    gathered = [torch.zeros_like(cs) for _ in range(world)]
    dist.all_gather(gathered, cs)
    out = {"replica_checksums": [[float(x) for x in g[:2].tolist()] for g in gathered],
           "replicas_identical": all(torch.equal(g[:3], gathered[0][:3]) for g in gathered),
           "arch_identical": all(torch.equal(g[2], gathered[0][2]) for g in gathered),
           # the clip norm of the last w-step: every rank computes it from the same averaged gradients
           "clip_norm_identical": all(torch.equal(g[3], gathered[0][3]) for g in gathered),
           "clip_norm": [float(g[3]) for g in gathered]}
    params = list(model.parameters())
    p_drop, model.dropout.p = model.dropout.p, 0.0
    try:
        for p_ in params:
            p_.grad = None
        batch = [t.to(dev) for t in synth_batch(5000 + rank, shard_batch, a.vocab, a.img)]
        loss = model._loss(*batch)
        loss.backward()
        grads = [p_.grad if p_.grad is not None else torch.zeros_like(p_) for p_ in params]
        reducer(grads)
        torch.cuda.synchronize()
    finally:
        model.dropout.p = p_drop
    if rank == 0:
        from oracle import pcdarts_oracle as O
        torch.set_num_threads(max(1, (os.cpu_count() or 1) - 1))
        t_oracle = time.time()
        sd = {k: v.detach().cpu().clone() for k, v in model.state_dict().items()}
        par, buf = O.split_state(sd)
        keys = [k for k, _ in model.named_parameters()]
        for v in par.values():
            v.requires_grad_(True)
        arch = [t.detach().cpu().clone() for t in model.arch_parameters()]
        acc = None
        for r in range(world):
            b = synth_batch(5000 + r, shard_batch, a.vocab, a.img)
            bns = O.BNState({k: v.clone() for k, v in buf.items()})
            l_r = O.vqa_loss(par, bns, arch, *b, dropout_p=0.0)
            g_r = torch.autograd.grad(l_r, [par[k] for k in keys], allow_unused=True)
            g_r = [torch.zeros_like(par[k]) if g is None else g for g, k in zip(g_r, keys)]
            acc = g_r if acc is None else [x + y for x, y in zip(acc, g_r)]
            if r == 0:
                out["rank0_loss_rel_err"] = abs(float(loss.detach()) - float(l_r.detach())) / abs(float(l_r.detach()))
        errs = []
        for k, g, ref in zip(keys, grads, acc):
            ref = ref / world
            den = float(ref.abs().max())
            errs.append((float((g.cpu() - ref).abs().max()) / den if den > 0 else float(g.abs().max()), k))
        errs.sort(reverse=True)
        out["averaged_grads_vs_oracle"] = {
            "tensors": len(errs), "share_within_1e-4": sum(e <= 1e-4 for e, _ in errs) / len(errs), "worst": errs[:3],
            "shards": world, "samples_per_shard": shard_batch, "oracle_seconds": round(time.time() - t_oracle, 1),
            "note": "search-net tensors beyond 1e-4 are ReLU / max-pool tie flips (~1/sqrt(B*H*W), DESIGN.md §2)"}
    dist.barrier(group=cpu_group) if cpu_group is not None else dist.barrier()
    return out


def gemm_roofline(a, dev):
    """Second roofline entry (tensor pipe): the vocabulary projection of one pass — M = B*30 rows, K = 512, N = V — through
    pcd_gemm_tn_3xtf32, algorithmic flops counted ONCE (the 3xTF32 split issues three MMAs per product), against the box's
    TF32 tensor throughput MEASURED here with a single-pass TF32 GEMM (torch.matmul, allow_tf32, 8192^3, best of 10)."""
    from pcd_ops import Linear3xTF32Function
    keep = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        x = torch.randn(8192, 8192, device=dev)
        y = torch.randn(8192, 8192, device=dev)
        best = 1e9
        for _ in range(10):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); torch.matmul(x, y); e1.record(); torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        peak = 2 * 8192 ** 3 / (best * 1e-3) / 1e12
    finally:
        torch.backends.cuda.matmul.allow_tf32 = keep
    del x, y
    M, K, Nn = a.batch * 30, DIMS["hidden_size"], a.vocab
    h = torch.randn(M, K, device=dev)
    w = torch.randn(Nn, K, device=dev) / K ** 0.5
    b = torch.zeros(Nn, device=dev)
    flush = torch.empty(64 << 20, dtype=torch.float32, device=dev)
    for _ in range(3):
        Linear3xTF32Function.apply(h, w, b)
    tot, iters = 0.0, 10
    for _ in range(iters):
        flush.zero_()                                   # L2 flush: the 36.6 MB weight matrix must come from HBM as in the step
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); Linear3xTF32Function.apply(h, w, b); e1.record(); torch.cuda.synchronize()
        tot += e0.elapsed_time(e1)
    ms = tot / iters
    achieved = 2.0 * M * Nn * K / (ms * 1e-3) / 1e12
    return {"bound": "tensor", "kernel": f"gemm_tn_3xtf32, vocabulary projection forward ({M} x {K} x {Nn})", "achieved": achieved,
            "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak, "ms": ms, "traffic": None,
            # what the tensor pipe actually executes: three TF32 MMAs per algorithmic product — the ceiling of `frac` is 1/3
            "executed_tflops": 3.0 * achieved, "executed_frac": 3.0 * achieved / peak,
            "peak_source": "measured in this run: torch.matmul fp32 with TF32 tensor cores, 8192^3, best of 10",
            "note": "algorithmic flops counted once; the kernel issues 3 tcgen05.mma.kind::tf32 per product (hi*hi + hi*lo + lo*hi)"}


def lct_alpha_step_bench(a, dev, iters=3):
    """ArchitectLct.step (basic_vqa/pcdarts/architect_lct.py:32-92) at the reference's default sizes: EF = PC-DARTS VqaModel on
    the kernels, W = VGG19 VqaModel (random weights: no download), B = 64, deterministic question sampling."""
    import config
    from architect_factory import get_architect
    from models import VqaModel as WModel
    from models_lct import VqaModel as EfModel
    config.ARCH_TYPE = "darts"
    torch.manual_seed(10)
    dims = dict(DIMS, qst_vocab_size=a.vocab)
    ef = EfModel(**dims).to(dev).train()
    w = WModel(pretrained=False, **dims).to(dev).train()
    arch = get_architect(ef, w, torch.optim.Adam(ef.parameters(), lr=1e-3), torch.optim.Adam(w.parameters(), lr=1e-3))
    tr = [t.to(dev) for t in synth_batch(10, a.batch, a.vocab, a.img)]
    va = [t.to(dev) for t in synth_batch(11, a.batch, a.vocab, a.img)]
    arch.step(*tr, *va, 1e-3, 1e-3)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        arch.step(*tr, *va, 1e-3, 1e-3)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / iters
    res = {"ms_per_alpha_step_eager": ms, "batch": a.batch, "w_val_loss": float(arch.last["unrolled_loss"]),
           "passes": "6 fwd + 5 bwd search-net, 3 greedy decodes, VGG19 W-model (stock torch) unroll + 2 HVP passes"}
    try:
        from search import GraphedLctStep
        g = GraphedLctStep(arch, tr, va, 1e-3, 1e-3)
        g()
        torch.cuda.synchronize()
        e0.record()
        for _ in range(iters):
            g()
        e1.record()
        torch.cuda.synchronize()
        ms_g = e0.elapsed_time(e1) / iters
        res.update(ms_per_alpha_step=ms_g, alpha_steps_per_s=1e3 / ms_g, mode="CUDA graph", w_val_loss_graph=float(g.loss))
    except Exception as e:
        res.update(ms_per_alpha_step=ms, alpha_steps_per_s=1e3 / ms, mode="eager (graph capture failed: %s)" % repr(e)[:160])
    return res


def mixedop_microbench(dev, B, hbm):
    """MixedOp fwd+bwd at the five production edge shapes (SURVEY.md §8d), L2 flushed between iterations."""
    from pcdarts.model_search import MixedOp
    flush = torch.empty(128 << 20, dtype=torch.float32, device=dev)
    res = []
    for name, C, s, H, count in EDGE_SHAPES:
        m = MixedOp(C, s).to(dev).train()
        x = torch.randn(B, C, H, H, device=dev, requires_grad=True)
        w = torch.softmax(torch.randn(8, device=dev), 0).requires_grad_(True)
        G = torch.randn(B, C, H // s, H // s, device=dev)
        for _ in range(3):
            m(x, w).backward(G)
        tot = 0.0
        iters = 5
        for _ in range(iters):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            m(x, w).backward(G)
            e1.record()
            torch.cuda.synchronize()
            tot += e0.elapsed_time(e1)
        ms = tot / iters
        c = C // 4
        s_in, s_out = B * H * H, B * (H // s) * (H // s)
        fwd = 4 * C * (s_in + s_out)
        bwd = 4 * s_in * (2 * C + c) if s == 1 else 4 * (C * s_out + 2 * C * s_in)
        gbs = (fwd + bwd) / 1e9 / (ms / 1e3)
        res.append({"shape": name, "edges_per_pass": count, "ms": ms, "algorithmic_mb": (fwd + bwd) / 1e6,
                    "gb_per_s": gbs, "frac_of_hbm_peak": gbs / hbm})
    return res


def derived_network_bench(model, dev, B=256, img=64):
    """BASELINE config 5 (SURVEY.md §8f-4): one training pass (forward + backward + SGD step) of the network DERIVED from the
    search network's current genotype (pcdarts/model.py, stand-alone op kernels on all channels) at a larger per-GPU batch."""
    from pcdarts.model import derive
    net = derive(model.img_encoder.darts).to(dev).train()
    opt = torch.optim.SGD(net.parameters(), lr=0.025, momentum=0.9, weight_decay=3e-4, foreach=True)
    x = torch.randn(B, 3, img, img, device=dev)
    G = torch.randn(B, net.output_ch * 49, device=dev)

    def step():
        opt.zero_grad(set_to_none=True)
        net(x).backward(G)
        opt.step()
    for _ in range(3):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    iters = 5
    e0.record()
    for _ in range(iters):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / iters
    return {"genotype_normal": [list(g) for g in net.genotype().normal], "genotype_reduce": [list(g) for g in net.genotype().reduce],
            "batch": B, "image": img, "ms_per_train_pass": ms, "images_per_s": B / (ms / 1e3),
            "weights": sum(p.numel() for p in net.parameters()),
            "note": "first versions of the op kernels (whole planes in shared memory, parity first); eager, no CUDA graph"}


def emit(obj):
    """The ONE JSON line, on the process's original stdout."""
    os.write(_REAL_STDOUT, (json.dumps(obj) + "\n").encode())


if __name__ == "__main__":
    args = parse()
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)              # NCCL's version banner and any library chatter: stderr, not the JSON channel
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)
