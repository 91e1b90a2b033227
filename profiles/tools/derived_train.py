"""Training the derived architecture as a VQA model (BASELINE config 5): the train step of a `derive_vqa` model at the benchmark
dimensions (64x64 images, V = 17858, 1000 answers, hidden 512, FlatAdam, clip 5), eager against GraphedTrainStep, at
drop_path_prob 0 and 0.2.  One process per GPU; prints one JSON line and writes it to --out.

    python profiles/tools/derived_train.py --batch 128 [--steps 20] [--out file.json]                 # one GPU
    torchrun --nproc_per_node 8 profiles/tools/derived_train.py --batch 128 --out file.json         # B = 1024 in all

--batch is per GPU.  Timing: CUDA events around `--steps` back-to-back steps after 3 warm-up steps, the slowest rank's time
under data parallelism.  Every arm starts from the same seeded model.  Under data parallelism every rank reports a float64
checksum of its weights and BatchNorm buffers after the arms ran; the replicas must agree.  With one process the drop-path
node kernel (pcd_droppath_sum_forward) is also timed alone at the first cell's shape (B = 128, C = 16, 64x64) over many
launches, against a device copy of the same tensor and against the stock composite (bernoulli_, div, mul_ per input, add).
The kernel's working set (3 x 33.5 MB) fits in the 126 MB L2, so neither number is an HBM rate; both sides run on the same
shape in the same process.
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

DIMS = dict(embed_size=512, ans_vocab_size=1000, word_embed_size=300, num_layers=1, hidden_size=512)


def card(index):
    name = torch.cuda.get_device_name(index)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits",
                              "-i", str(index)], capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        return {"name": name, "power_limit_w": float(out[0]), "sm_max_mhz": float(out[1])}
    except Exception as e:
        return {"name": name, "power_limit_w": None, "error": str(e)}


def batch(seed, B, V, dev):
    g = torch.Generator().manual_seed(seed)
    img = torch.randn(B, 3, 64, 64, generator=g)
    qst = torch.randint(0, V, (B, 30), generator=g)
    qst[:, 0] = 2
    return [img.to(dev), qst.to(dev), torch.randint(0, 1000, (B,), generator=g).to(dev)]


def events_ms(fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def node_kernel(dev, B=128, C=16, H=64, iters=200):
    from pcd_ops import droppath_sum
    h1, h2 = torch.randn(B, C, H, H, device=dev), torch.randn(B, C, H, H, device=dev)
    keep = torch.full((1,), 0.8, device=dev)
    seed = torch.randint(0, 2 ** 62, (1,), device=dev)
    dst = torch.empty_like(h1)
    kernel = lambda: droppath_sum(h1, h2, True, True, keep, seed, 0, 0)
    copy_ = lambda: dst.copy_(h1)
    mask = torch.empty(B, 1, 1, 1, device=dev)

    def stock():        # DARTS's drop_path on both inputs, then the node's add
        a = h1.div(0.8).mul_(mask.bernoulli_(0.8))
        b = h2.div(0.8).mul_(mask.bernoulli_(0.8))
        return a + b
    res = {}
    nbytes = h1.numel() * 4
    for name, fn, traffic in (("kernel", kernel, 3 * nbytes), ("copy", copy_, 2 * nbytes), ("stock_composite", stock, 3 * nbytes)):
        for _ in range(10):
            fn()
        ms = min(events_ms(fn, iters) for _ in range(3)) / iters
        res[name] = {"us_per_call": 1e3 * ms, "gb_per_s_on_3_tensors" if name != "copy" else "gb_per_s":
                     traffic / (ms / 1e3) / 1e9}
    res["shape"] = [B, C, H, H]
    res["kernel_over_copy_bandwidth"] = res["kernel"]["gb_per_s_on_3_tensors"] / res["copy"]["gb_per_s"]
    res["stock_over_kernel_time"] = res["stock_composite"]["us_per_call"] / res["kernel"]["us_per_call"]
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=128, help="per GPU")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--vocab", type=int, default=17858)
    ap.add_argument("--out")
    a = ap.parse_args()
    import torch.distributed as dist
    import pcd_dist
    import pcd_flat
    import pcd_native
    from search import GraphedTrainStep, SearchStep
    from vqa_model import VqaModel, derive_vqa
    rank, world = pcd_dist.init_from_env()
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    lib = pcd_native.load_cuda()
    torch.manual_seed(10)
    search = VqaModel(qst_vocab_size=a.vocab, img_encoder_type="darts", **DIMS).to(dev).train()
    torch.manual_seed(11)
    base = derive_vqa(search)
    del search
    reducer = pcd_dist.GradReducer() if world > 1 else None
    if world > 1:
        for t in list(base.parameters()) + list(base.buffers()):
            dist.broadcast(t.data, 0)
    data = batch(100 + rank, a.batch, a.vocab, dev)
    arms = {}
    for p in (0.0, 0.2):
        for mode in ("eager", "graph"):
            torch.manual_seed(1234)          # one drop-path seed stream on every rank
            model = copy.deepcopy(base)
            model.img_encoder.darts.drop_path_prob = p
            step = SearchStep(model, None, pcd_flat.FlatAdam(model.parameters(), lr=1e-3), reducer=reducer, grad_clip=5.0)
            if mode == "graph":
                g = GraphedTrainStep(step, data)
                fn = g
            else:
                fn = lambda: step.w_step(*data)
            losses = [float(fn()) for _ in range(3)]
            l0 = lib.pcd_launch_count()
            ms = events_ms(fn, a.steps)
            launches = (lib.pcd_launch_count() - l0) / a.steps
            t = torch.tensor([ms], device=dev)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t) / a.steps
            with torch.no_grad():
                ck = torch.stack([x.detach().double().sum() for x in list(model.parameters()) + list(model.buffers())
                                  if x.is_floating_point()]).sum()
            cks = [torch.zeros_like(ck) for _ in range(world)]
            if world > 1:
                dist.all_gather(cks, ck)
            else:
                cks = [ck]
            arms[f"{mode}_p{p}"] = {"ms_per_step": ms, "steps_per_s": 1e3 / ms, "images_per_s": world * a.batch * 1e3 / ms,
                                    "warmup_losses": losses, "library_launches_per_step": launches if mode == "eager" else None,
                                    "replica_checksums": [float(c) for c in cks],
                                    "replicas_identical": len({float(c) for c in cks}) == 1}
            del fn, step, model
            if mode == "graph":
                del g
            torch.cuda.empty_cache()
    out = {"workload": "derive_vqa(VqaModel(512, V, 1000, 300, 1, 512)) train step: w_step, FlatAdam lr 1e-3, clip 5, 64x64",
           "vocab": a.vocab, "batch_per_gpu": a.batch, "global_batch": world * a.batch, "gpus": world,
           "steps_timed": a.steps, "arms": arms}
    for p in ("0.0", "0.2"):
        out[f"graph_speedup_p{p}"] = arms[f"eager_p{p}"]["ms_per_step"] / arms[f"graph_p{p}"]["ms_per_step"]
    if world == 1:
        out["node_kernel"] = node_kernel(dev)
    if rank == 0:
        out["card"] = card(local)
        line = json.dumps(out)
        print(line)
        if a.out:
            with open(a.out, "w") as f:
                f.write(line + "\n")
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
