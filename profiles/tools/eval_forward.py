"""Eval-mode forward (BatchNorm from running statistics) of the search network and of a VqaModel validation batch, against
the two nearest alternatives, in one run on one GPU.  Prints one JSON line.

    python profiles/tools/eval_forward.py [--iters N] [--out file.json]

Arms (search network, 64 x 64 input, B = 64 and 256):
  eval          Network.eval() under torch.no_grad(): eval stem, eval preprocess, one launch per node
  train_nograd  the native training-mode forward under torch.no_grad() (what ran before eval mode existed; it also updates
                the running statistics, so it runs on a copy)
  stock_eval    oracle.network_forward(..., training=False): stock ATen / cuDNN eval forward on the same GPU (fp32, TF32 off)
Every timed iteration is preceded by a write of 512 MB (larger than the 126 MB L2), outside the timed events.
Bytes are computed from shapes for the eval forward (stem read + write; per cell the two input states read and the two
preprocessed states written; every edge reads its whole source state once; every node is written once; global pooling
reads the last cell), and set against a device-to-device copy bandwidth measured in the same run.
VqaModel validation batch at the benchmark dimensions (hidden 512, word embedding 300, 1000 answers, V = 17858, B = 64):
forward + _loss (what a validation loop runs per batch) and generate().
"""
import argparse
import copy
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path[:0] = [os.path.join(ROOT, "lct-vqa_b200"), ROOT, os.path.join(ROOT, "tests")]


def card():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        return {"name": name, "power_limit_w": float(out[0]), "sm_max_mhz": float(out[1])}
    except Exception as e:           # the number stays usable; say why the power limit is missing
        return {"name": name, "power_limit_w": None, "error": str(e)}


class Timer:
    def __init__(self):
        self.flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")

    def __call__(self, fn, iters, warmup=3):
        for _ in range(warmup):
            fn()
        ts = []
        for _ in range(iters):
            self.flush.fill_(1)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            b.synchronize()
            ts.append(a.elapsed_time(b))
        ts.sort()
        return {"ms_median": ts[len(ts) // 2], "ms_min": ts[0], "ms_max": ts[-1], "iters": iters}


def copy_bandwidth(timer):
    src = torch.empty(1 << 30, dtype=torch.uint8, device="cuda")
    dst = torch.empty_like(src)
    t = timer(lambda: dst.copy_(src), 10)
    return 2 * src.numel() / (t["ms_median"] * 1e-3)


def eval_bytes(B, H, C=16, layers=4):
    from oracle import pcdarts_oracle as O
    f = 4
    total = B * 3 * H * H * f + B * 3 * C * H * H * f                    # stem
    h = H
    for cpp, cp, c, red, rp in O.cell_plan(C, layers):
        h0 = 2 * h if rp else h
        ho = h // 2 if red else h
        total += B * (cpp * h0 * h0 + cp * h * h) * f + 2 * B * c * h * h * f          # preprocess
        for i in range(4):
            for j in range(2 + i):
                total += B * c * (h * h if j < 2 else ho * ho) * f          # each edge reads its source state once
            total += B * c * ho * ho * f                                    # node written once
        h = ho
    total += B * 4 * 64 * h * h * f + B * 256 * 49 * f                      # global pooling
    return total


def network_arms(B, H, iters, timer, bw):
    import config
    import parity_cases as P
    from oracle import pcdarts_oracle as O
    perms = {}

    def shuffle(x, groups=4):        # the oracle's channel shuffle with its index cached on the GPU
        key = (x.shape[1], groups, x.device)
        if key not in perms:
            perms[key] = torch.from_numpy(O.shuffle_perm(x.shape[1], groups)).to(x.device)
        return x.index_select(1, perms[key])

    O.channel_shuffle = shuffle
    config.DEVICE = "cuda"
    from pcdarts.model_search import Network
    net = Network(16, 10, 4)
    P._fill(net, 17)
    net.cuda()
    x = torch.randn(B, 3, H, H, device="cuda")
    twin = copy.deepcopy(net).train()
    net.eval()
    res = {}
    with torch.no_grad():
        res["eval"] = timer(lambda: net(x), iters)
        res["train_nograd"] = timer(lambda: twin(x), iters)
        par, buf = O.split_state({k: v.detach() for k, v in net.state_dict().items()})
        arch = [a.detach() for a in net.arch_parameters()]
        res["stock_eval"] = timer(lambda: O.network_forward(par, O.BNState(buf), arch, x, training=False), iters)
        y, yr = net(x), O.network_forward(par, O.BNState(buf), arch, x, training=False)
        res["eval_vs_stock_rel_err"] = ((y - yr).norm() / yr.norm()).item()
    nbytes = eval_bytes(B, H)
    for k in ("eval", "train_nograd", "stock_eval"):
        res[k]["images_per_s"] = B / (res[k]["ms_median"] * 1e-3)
    res["eval_bytes"] = nbytes
    res["eval_hbm_frac"] = nbytes / (res["eval"]["ms_median"] * 1e-3) / bw
    res["speedup_vs_train_nograd"] = res["train_nograd"]["ms_median"] / res["eval"]["ms_median"]
    res["speedup_vs_stock_eval"] = res["stock_eval"]["ms_median"] / res["eval"]["ms_median"]
    # kernel split of one eval forward (CUDA events around every launch, a separate pass)
    import pcd_native
    lib = pcd_native.load_cuda()
    lib.pcd_profile_enable(1)
    with torch.no_grad():
        net(x)
    torch.cuda.synchronize()
    res["eval_kernels_ms"] = {k: round(v[0], 4) for k, v in pcd_native.profile_collect(lib).items()}
    lib.pcd_profile_enable(0)
    return res


def vqa_arms(iters, timer):
    import config
    import parity_cases as P
    config.DEVICE = "cuda"
    from vqa_model import VqaModel
    V = 17858
    m = VqaModel(img_encoder_type="darts", qst_vocab_size=V, **P.FULL_DIMS)
    P._fill(m, 400)
    m.cuda().eval()
    img, qst, lbl = (t.cuda() for t in P.full_batch(5, 64, V, 64))

    def val_step():
        m(img, qst)
        m._loss(img, qst, lbl)

    with torch.no_grad():
        return {"forward_plus_loss": timer(val_step, iters), "generate": timer(lambda: m.generate(img), iters)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("eval_forward.py measures on a GPU; none is visible")
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    timer = Timer()
    bw = copy_bandwidth(timer)
    rec = {"metric": "eval_forward", "card": card(), "copy_bandwidth_gb_s": bw / 1e9, "input": "64x64",
           "network": {str(B): network_arms(B, 64, a.iters, timer, bw) for B in (64, 256)},
           "vqa_validation_batch_b64": vqa_arms(a.iters, timer)}
    line = json.dumps(rec)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
