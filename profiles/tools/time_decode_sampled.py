"""QstEncoder.generate at the production size (B = 64, H = 512, E = 300, V = 17858, T = 30, temperature 0.1), three arms in one
run on one GPU.  Prints one JSON line.

    python profiles/tools/time_decode_sampled.py [--calls N] [--out file.json]

Arms:
  greedy_kernel   deterministic=True: pcd_decode in greedy mode, one persistent cooperative launch
  sampled_kernel  deterministic=False: pcd_decode in sampled mode (the same kernel, Gumbel-max on Philox noise) + the seed draw
  stock_sampled   deterministic=None: the reference's module loop (nn.LSTM step, Linear, softmax, torch.multinomial per word),
                  which is what deterministic=False ran before the sampled kernel existed
Timing: CUDA events around blocks of back-to-back calls, the arms alternating block by block, after warm-up; per-call time
per block, median / min / max over the blocks.  No cache flush: W_out (36.6 MB) and the LSTM weights stay L2-resident between
calls, as they are between the three decodes inside an LCT alpha-step.  A separate torch.profiler pass per arm gives the
per-kernel device time of one call.
"""
import argparse
import collections
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path[:0] = [os.path.join(ROOT, "lct-vqa_b200"), ROOT]


def card():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        return {"name": name, "power_limit_w": float(out[0]), "sm_max_mhz": float(out[1])}
    except Exception as e:           # the number stays usable; say why the power limit is missing
        return {"name": name, "power_limit_w": None, "error": str(e)}


def kernel_breakdown(fn, calls=3):
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            fn()
        torch.cuda.synchronize()
    agg = collections.defaultdict(lambda: [0.0, 0])
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA:
            agg[e.name][0] += e.device_time
            agg[e.name][1] += 1
    rows = sorted(agg.items(), key=lambda kv: -kv[1][0])
    return {"kernel_ms_per_call": sum(v[0] for _, v in rows) / 1e3 / calls,
            "launches_per_call": sum(v[1] for _, v in rows) / calls,
            "top": [{"kernel": k[:120], "ms_per_call": v[0] / 1e3 / calls, "launches_per_call": v[1] / calls} for k, v in rows[:6]]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=200, help="timed calls per arm (>= 100)")
    ap.add_argument("--block", type=int, default=20, help="back-to-back calls per timed block")
    ap.add_argument("--out")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_decode_sampled.py measures on a GPU; none is visible")
    from vqa_model import QstEncoder
    B, H, E, V, T, temperature = 64, 512, 300, 17858, 30, 0.1
    torch.manual_seed(0)
    q = QstEncoder(V, E, H, 1, H, temperature=temperature, max_length=T).to("cuda")
    img = torch.randn(B, H, device="cuda") * 0.1

    def arm(mode):
        def run():
            q.deterministic = mode
            return q.generate(img)
        return run

    arms = {"greedy_kernel": arm(True), "sampled_kernel": arm(False), "stock_sampled": arm(None)}
    for fn in arms.values():
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    per_call = {k: [] for k in arms}
    for _ in range(max(1, (a.calls + a.block - 1) // a.block)):
        for name, fn in arms.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(a.block):
                fn()
            e1.record()
            e1.synchronize()
            per_call[name].append(e0.elapsed_time(e1) / a.block)
    res = {}
    for name, ts in per_call.items():
        s = sorted(ts)
        res[name] = {"ms_per_call_median": s[len(s) // 2], "ms_per_call_min": s[0], "ms_per_call_max": s[-1],
                     "calls": len(ts) * a.block, "profiler": kernel_breakdown(arms[name])}
    g, smp, st = (res[k]["ms_per_call_median"] for k in ("greedy_kernel", "sampled_kernel", "stock_sampled"))
    rec = {"metric": "decode_sampled", "card": card(), "shape": dict(B=B, H=H, E=E, V=V, T=T, temperature=temperature),
           "l2": "no flush: W_out (36.6 MB) stays L2-resident between calls, as inside an LCT alpha-step",
           "timing": f"CUDA events over blocks of {a.block} back-to-back calls, arms alternating, median over blocks",
           "arms": res, "sampled_over_greedy": smp / g - 1.0, "stock_sampled_over_sampled_kernel": st / smp}
    line = json.dumps(rec)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
