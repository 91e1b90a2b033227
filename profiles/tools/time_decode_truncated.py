"""Truncated sampling in QstEncoder.generate at the production size (B = 64, H = 512, E = 300, V = 17858, T = 30), at
temperatures 0.1 and 1.0, five arms in one run on one GPU.  Prints one JSON line.

    python profiles/tools/time_decode_truncated.py [--calls N] [--out file.json]

Arms (per temperature):
  sampled        untruncated sampling: pcd_decode in sampled mode (Gumbel-max in the phase-B epilogue) + the seed draw
  top_k50        pcd_decode in sampled mode with truncate = 1, top_k = 50: logits kept in the workspace, one more grid barrier
                 and a radix select per row and step
  top_p0.9       the same with top_p = 0.9
  top_k50_p0.9   both
  stock_k50_p0.9 a stock-torch loop (nn.LSTM step, Linear, topk, sorted cumsum, softmax, torch.multinomial per word) doing
                 the same filtering: what a user had to write before the kernel took top_k / top_p
Timing: CUDA events around blocks of back-to-back calls, the arms alternating block by block, after warm-up; per-call time
per block, median / min / max over the blocks.  No cache flush: W_out (36.6 MB) and the LSTM weights stay L2-resident between
calls, as they are between the three decodes inside an LCT alpha-step.
"""
import argparse
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


def stock_truncated(q, img, temperature, top_k, top_p):
    """The module loop of QstEncoder.generate with HF-style filtering: temperature, top-k, then top-p over the top-k set."""
    B = img.shape[0]
    h = img.view(1, B, -1)
    state = (h, h)
    word = torch.full((B, 1), 2, dtype=torch.long, device=img.device)
    current = q.tanh(q.word2vec(word)).transpose(0, 1)
    qst = torch.zeros((B, q.max_length), dtype=torch.long, device=img.device)
    for t in range(q.max_length):
        out, state = q.lstm(current, state)
        logits = q.fc1(q.tanh(out[0])) / temperature
        val, idx = torch.topk(logits, top_k, dim=1)                      # sorted, descending
        prob = torch.softmax(val, dim=1)
        drop = prob.cumsum(1) - prob >= top_p                           # keep the shortest prefix reaching top_p
        prob = prob.masked_fill(drop, 0.0)
        pick = idx.gather(1, torch.multinomial(prob, 1))
        current = q.word2vec(pick).transpose(0, 1)
        qst[:, t] = pick[:, 0]
    return qst


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=200, help="timed calls per arm and temperature (>= 100)")
    ap.add_argument("--block", type=int, default=20, help="back-to-back calls per timed block")
    ap.add_argument("--out")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_decode_truncated.py measures on a GPU; none is visible")
    torch.backends.cuda.matmul.allow_tf32 = False
    from vqa_model import QstEncoder
    B, H, E, V, T = 64, 512, 300, 17858, 30
    torch.manual_seed(0)
    q = QstEncoder(V, E, H, 1, H, deterministic=False, max_length=T).to("cuda")
    img = torch.randn(B, H, device="cuda") * 0.1
    res = {}
    for temperature in (0.1, 1.0):
        def arm(top_k, top_p):
            def run():
                q.temperature, q.top_k, q.top_p = temperature, top_k, top_p
                return q.generate(img)
            return run

        def stock():
            with torch.no_grad():
                return stock_truncated(q, img, temperature, 50, 0.9)

        arms = {"sampled": arm(0, 1.0), "top_k50": arm(50, 1.0), "top_p0.9": arm(0, 0.9), "top_k50_p0.9": arm(50, 0.9),
                "stock_k50_p0.9": stock}
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
        r = {}
        for name, ts in per_call.items():
            s = sorted(ts)
            r[name] = {"ms_per_call_median": s[len(s) // 2], "ms_per_call_min": s[0], "ms_per_call_max": s[-1],
                       "calls": len(ts) * a.block}
        med = {k: v["ms_per_call_median"] for k, v in r.items()}
        r["over_sampled"] = {k: med[k] / med["sampled"] - 1.0 for k in ("top_k50", "top_p0.9", "top_k50_p0.9")}
        r["stock_over_kernel_k50_p0.9"] = med["stock_k50_p0.9"] / med["top_k50_p0.9"]
        res[f"temperature_{temperature}"] = r
    rec = {"metric": "decode_truncated", "card": card(), "shape": dict(B=B, H=H, E=E, V=V, T=T),
           "l2": "no flush: W_out (36.6 MB) stays L2-resident between calls, as inside an LCT alpha-step",
           "timing": f"CUDA events over blocks of {a.block} back-to-back calls, arms alternating, median over blocks",
           "stock_arm": "nn.LSTM step + Linear + topk + softmax + sorted cumsum + multinomial per word, TF32 off",
           "results": res}
    line = json.dumps(rec)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
