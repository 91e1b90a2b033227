"""End-of-sequence decoding at the production size (B = 64, H = 512, E = 300, V = 17858, T = 30): greedy, sampled and beam
(K = 4) with end_token against the same calls without it, all in one run on one GPU.  Prints one JSON line and writes it
to --out.

    python profiles/tools/time_decode_stop.py [--calls N] [--out profiles/decode_stop.json]

Model: a synthetic decoder (scaled random weights, so that the log-probabilities are far from uniform as in a trained one)
whose <end> (index 3) output bias is raised until the greedy rows end at a spread of lengths: the smallest bias in the sweep
whose median greedy length is at most --target-median.  The lengths every arm produced are recorded.
Timing: CUDA events around blocks of back-to-back calls, the arms alternating block by block, after warm-up; per-call time
per block, median / min / max over the blocks.  No cache flush: W_out (36.6 MB) stays L2-resident between calls, as it does
between the decodes inside an LCT alpha-step.  A launch's time is expected to follow its longest row, not the mean length.
Early exit: the stopped greedy and beam calls also run on two copies of the projection, one whose <end> bias (50) ends every
row at step 0 and one whose bias (-1e4) never lets <end> be chosen; their time ratio shows whether the kernel leaves its
time loop once every row has finished.
"""
import argparse
import copy
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path[:0] = [os.path.join(ROOT, "lct-vqa_b200"), ROOT]

END, PAD = 3, 0


def card():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader,nounits",
                              "-i", "0"], capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        return {"name": name, "power_limit_w": float(out[0]), "sm_mhz": float(out[1]), "sm_max_mhz": float(out[2])}
    except Exception as e:           # the number stays usable; say why the power limit is missing
        return {"name": name, "power_limit_w": None, "error": str(e)}


def synthetic_decoder(B, H, E, V, seed=0):
    g = torch.Generator().manual_seed(seed)
    emb, lstm, proj = torch.nn.Embedding(V, E), torch.nn.LSTM(E, H, 1), torch.nn.Linear(H, V)
    with torch.no_grad():
        for p in list(emb.parameters()) + list(lstm.parameters()) + list(proj.parameters()):
            p.copy_(torch.randn(p.shape, generator=g) * (0.5 if p.dim() > 1 else 0.1) / (p.shape[-1] ** 0.5 if p.dim() > 1 else 1.0))
        emb.weight.mul_(E ** 0.5)
        proj.weight.mul_(6.0)
    h0 = torch.randn(B, H, generator=g) * 0.5
    return [m.to("cuda") for m in (emb, lstm, proj)], h0.to("cuda")


def lengths(tokens, T):
    """Length of each row counting the first <end> (T where there is none)."""
    hit = tokens == END
    return torch.where(hit.any(-1), hit.long().argmax(-1) + 1, torch.full(tokens.shape[:-1], T, device=tokens.device))


def histogram(ls):
    ls = sorted(int(x) for x in ls)
    return {"min": ls[0], "median": ls[len(ls) // 2], "max": ls[-1], "mean": sum(ls) / len(ls), "values": ls}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=100, help="timed calls per arm")
    ap.add_argument("--block", type=int, default=10, help="back-to-back calls per timed block")
    ap.add_argument("--target-median", type=int, default=10, help="median greedy length the <end> bias is raised to")
    ap.add_argument("--out")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_decode_stop.py measures on a GPU; none is visible")
    from pcd_ops import decode_beam, decode_greedy, decode_sample
    B, H, E, V, T, K = 64, 512, 300, 17858, 30, 4
    (emb, lstm, proj), img = synthetic_decoder(B, H, E, V)
    sweep = []
    for bias in [0.5 * i for i in range(41)]:
        with torch.no_grad():
            proj.bias[END] = bias
        med = int(lengths(decode_greedy(img, lstm, emb, proj, T), T).median())
        sweep.append((bias, med))
        if med <= a.target_median:
            break
    end_bias = sweep[-1][0]
    seed = 1234
    proj_at0, proj_never = copy.deepcopy(proj), copy.deepcopy(proj)
    with torch.no_grad():
        proj_at0.bias[END] = 50.0
        proj_never.bias[END] = -1e4
    arms = {
        "greedy": lambda: decode_greedy(img, lstm, emb, proj, T),
        "greedy_stop": lambda: decode_greedy(img, lstm, emb, proj, T, end_token=END, pad_token=PAD),
        "sampled": lambda: decode_sample(img, lstm, emb, proj, T, 1.0, seed=seed),
        "sampled_stop": lambda: decode_sample(img, lstm, emb, proj, T, 1.0, seed=seed, end_token=END, pad_token=PAD),
        f"beam{K}": lambda: decode_beam(img, lstm, emb, proj, T, K),
        f"beam{K}_stop": lambda: decode_beam(img, lstm, emb, proj, T, K, end_token=END, pad_token=PAD),
        "greedy_stop_end_at_step0": lambda: decode_greedy(img, lstm, emb, proj_at0, T, end_token=END, pad_token=PAD),
        "greedy_stop_never_ends": lambda: decode_greedy(img, lstm, emb, proj_never, T, end_token=END, pad_token=PAD),
        f"beam{K}_stop_end_at_step0": lambda: decode_beam(img, lstm, emb, proj_at0, T, K, end_token=END, pad_token=PAD),
        f"beam{K}_stop_never_ends": lambda: decode_beam(img, lstm, emb, proj_never, T, K, end_token=END, pad_token=PAD),
    }
    for fn in arms.values():
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    dist = {"greedy": histogram(lengths(arms["greedy_stop"](), T).tolist()),
            "sampled": histogram(lengths(arms["sampled_stop"](), T).tolist())}
    bt = arms[f"beam{K}_stop"]()[0]
    dist[f"beam{K}_best"] = histogram(lengths(bt[:, 0], T).tolist())
    dist[f"beam{K}_longest_per_launch"] = [int(lengths(bt[i:i + 64 // K], T).max()) for i in range(0, B, 64 // K)]
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
                     "calls": len(ts) * a.block}
    med = {k: v["ms_per_call_median"] for k, v in res.items()}
    rec = {"metric": "decode_stop", "card": card(), "shape": dict(B=B, H=H, E=E, V=V, T=T, K=K),
           "model": f"synthetic decoder (scaled random weights, seed 0), <end> = {END} output bias {end_bias}",
           "end_bias_sweep": sweep, "lengths": dist,
           "l2": "no flush: W_out (36.6 MB) stays L2-resident between calls, as inside an LCT alpha-step",
           "timing": f"CUDA events over blocks of {a.block} back-to-back calls, arms alternating, median over blocks",
           "arms": res,
           "stop_over_full": {m: med[f"{m}_stop"] / med[m] for m in ("greedy", "sampled", f"beam{K}")},
           "early_exit_over_never_ends": {m: med[f"{m}_stop_end_at_step0"] / med[f"{m}_stop_never_ends"]
                                          for m in ("greedy", f"beam{K}")},
           "longest_row_over_T": {m: dist[m]["max"] / T for m in ("greedy", "sampled")}}
    line = json.dumps(rec)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
