"""Beam-search question decode at the production size (B = 64, H = 512, E = 300, V = 17858, T = 30), K in {1, 2, 4, 8}, against
the greedy kernel and a stock-torch beam loop, all in one run on one GPU.  Prints one JSON line and writes it to --out.

    python profiles/tools/time_decode_beam.py [--calls N] [--out profiles/decode_beam.json]

Arms:
  greedy_kernel   pcd_decode in greedy mode (QstEncoder.generate with beam_size = 1): one persistent cooperative launch
  beam_kernel_K   pcd_ops.decode_beam(..., K): ceil(64 K / 64) launches of the persistent kernel in beam mode
  stock_beam_K    the loop a user would write without the kernel: per word an nn.LSTM step, Linear(H, V) over B K rows,
                  log_softmax, topk over K V candidates per item and a gather of the parents' states; TF32 off
Timing: CUDA events around blocks of back-to-back calls, the arms alternating block by block, after warm-up; per-call time
per block, median / min / max over the blocks.  No cache flush: W_out (36.6 MB) stays L2-resident between calls, as it does
between the decodes inside an LCT alpha-step.  `stock_agrees` is the share of items whose best beam has the kernel's words.
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
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader,nounits",
                              "-i", "0"], capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        return {"name": name, "power_limit_w": float(out[0]), "sm_mhz": float(out[1]), "sm_max_mhz": float(out[2])}
    except Exception as e:           # the number stays usable; say why the power limit is missing
        return {"name": name, "power_limit_w": None, "error": str(e)}


@torch.no_grad()
def stock_beam(q, img, K, T, start_token=2):
    """(tokens (B, K, T), scores (B, K)) by stock torch ops, the semantics of pcd_decode in beam mode."""
    B, H = img.shape
    V = q.fc1.out_features
    R = B * K
    h = img.repeat_interleave(K, 0)[None].contiguous()
    c = h.clone()
    x = torch.tanh(q.word2vec.weight[start_token]).expand(1, R, -1)
    s = torch.full((B, K), float("-inf"), device=img.device)
    s[:, 0] = 0.0
    base = torch.arange(B, device=img.device)[:, None] * K
    words, parents = [], []
    for _ in range(T):
        out, (h, c) = q.lstm(x, (h, c))
        lam = torch.log_softmax(q.fc1(torch.tanh(out[0])), dim=1)
        s, idx = (s.reshape(R, 1) + lam).reshape(B, K * V).topk(K, dim=1)
        k, v = idx // V, idx % V
        rows = (base + k).reshape(R)
        h, c = h[:, rows], c[:, rows]
        x = q.word2vec(v.reshape(1, R))
        words.append(v); parents.append(k)
    tokens = torch.empty(B, K, T, dtype=torch.long, device=img.device)
    cur = torch.arange(K, device=img.device).expand(B, K)
    for t in range(T - 1, -1, -1):
        tokens[:, :, t] = words[t].gather(1, cur)
        cur = parents[t].gather(1, cur)
    return tokens, s


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=100, help="timed calls per arm")
    ap.add_argument("--block", type=int, default=10, help="back-to-back calls per timed block")
    ap.add_argument("--out")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_decode_beam.py measures on a GPU; none is visible")
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    from pcd_ops import decode_beam, decode_greedy
    from vqa_model import QstEncoder
    B, H, E, V, T, widths = 64, 512, 300, 17858, 30, (1, 2, 4, 8)
    torch.manual_seed(0)
    q = QstEncoder(V, E, H, 1, H, max_length=T).to("cuda").eval()
    img = torch.randn(B, H, device="cuda") * 0.1
    arms = {"greedy_kernel": lambda: decode_greedy(img, q.lstm, q.word2vec, q.fc1, T)}
    for K in widths:
        arms[f"beam_kernel_{K}"] = (lambda K=K: decode_beam(img, q.lstm, q.word2vec, q.fc1, T, K))
        arms[f"stock_beam_{K}"] = (lambda K=K: stock_beam(q, img, K, T))
    for fn in arms.values():
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    agree = {}
    for K in widths:
        kt, _ = arms[f"beam_kernel_{K}"]()
        st, _ = arms[f"stock_beam_{K}"]()
        agree[K] = (kt[:, 0] == st[:, 0]).all(1).double().mean().item()
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
    rec = {"metric": "decode_beam", "card": card(), "shape": dict(B=B, H=H, E=E, V=V, T=T),
           "l2": "no flush: W_out (36.6 MB) stays L2-resident between calls, as inside an LCT alpha-step",
           "timing": f"CUDA events over blocks of {a.block} back-to-back calls, arms alternating, median over blocks",
           "tf32": False, "arms": res,
           "beam_over_greedy": {K: med[f"beam_kernel_{K}"] / med["greedy_kernel"] for K in widths},
           "stock_over_kernel": {K: med[f"stock_beam_{K}"] / med[f"beam_kernel_{K}"] for K in widths},
           "stock_agrees": agree}
    line = json.dumps(rec)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
