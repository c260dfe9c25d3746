"""Cost of the number of mixture components on cfg4's network (784-512-512, z 64, batch 16 384, bf16, objective R), measured
the way bench.py measures: graph replay of the whole training step, L2 flushed (256 MB write) between timed steps, CUDA events,
median over --steps per repeat.  Per K: samples/s and ms/step per repeat, FLOP/sample from shapes (bench.flops_per_sample), the
per-class device time of three eager steps (gmvae_profile_*), and, from torch.profiler in a run of its own, the device time of
the q(y|x) head kernels beside their HBM bytes (from shapes) and the time those bytes take at --copy-peak.

    python tools/bench_wide_k.py --out profiles/wide_k/cfg4_k.json
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from bench import WORKLOADS, flops_per_sample, synthetic_images  # noqa: E402
from tools.bench_deterministic import card, timed  # noqa: E402

HEAD_KERNELS = ("head_y_wide_fwd_kernel", "head_y_wide_bwd_kernel", "head_y_fwd_kernel", "head_y_bwd_kernel",
                "head_y_fwd_row_kernel", "head_y_bwd_row_kernel")


def head_bytes(B, K):
    """HBM bytes of the two q(y|x) head kernels of one step.  Forward: reads logits and Gumbel noise (fp32), writes y in fp32 and
    as the zero-padded bf16 operand row.  Backward: reads logits, y and dy (fp32), writes dlogits as the padded bf16 row."""
    Kp = (K + 7) // 8 * 8
    return {"fwd": B * K * 4 * 3 + B * Kp * 2, "bwd": B * K * 4 * 3 + B * Kp * 2}


def head_kernel_ms(eng, x, side, steps=3):
    from torch.profiler import ProfilerActivity, profile
    with torch.cuda.stream(side):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(steps):
                eng.train_step(x)
            side.synchronize()
    per = {}
    for ev in prof.key_averages():
        for tag in HEAD_KERNELS:
            if tag + "<" in ev.key or tag + "(" in ev.key:
                t = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0)   # us
                per[tag] = per.get(tag, 0.0) + t / 1e3 / steps
    return per


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ks", default="10,128,129,256,512,1024")
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--copy-peak", type=float, default=6533.0, help="GB/s, the measured device-to-device copy peak")
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    import gmvae_b200
    dev = torch.device("cuda", 0)
    side = torch.cuda.Stream(dev)
    l2 = torch.zeros(64 * 1024 * 1024, dtype=torch.float32, device=dev)
    base = WORKLOADS["cfg4"]
    B = base["batch"]
    x = synthetic_images(B, 1234).to(dev)
    res = {"card": card(), "workload": "cfg4 network (784-512-512, z 64), batch 16384, bf16, objective R; K varies",
           "method": "graph replay, L2 flushed between timed steps, CUDA events, median of --steps per repeat",
           "copy_peak_GBps": args.copy_peak, "ks": {}}
    for K in (int(k) for k in args.ks.split(",")):
        w = dict(base, mixture_components=K)
        eng = gmvae_b200.Engine(model="gmvae", data_size=784, latent_size=w["latent_size"], hidden_sizes=w["hidden_sizes"],
                                mixture_components=K, max_batch=B, seed=1234)
        with torch.cuda.stream(side):
            for _ in range(3):
                eng.train_step(x)
            eng.capture_step(x)
            for _ in range(5):
                eng.replay()
        side.synchronize()
        reps = []
        for _ in range(args.repeats):
            ms = timed(eng, eng.replay, args.steps, l2, side)
            reps.append({"ms_per_step": ms, "samples_per_s": B / ms * 1e3})
        with torch.cuda.stream(side):
            eng.profile(True)
            for _ in range(3):
                l2.add_(1)
                eng.train_step(x)
            side.synchronize()
            classes = {k: v["ms"] / 3 for k, v in eng.profile_read().items()}
            eng.profile(False)
        kern = head_kernel_ms(eng, x, side)
        eng.close()
        hb = head_bytes(B, K)
        floor = {k: v / (args.copy_peak * 1e9) * 1e3 for k, v in hb.items()}
        rec = {"repeats": reps, "flop_per_sample": flops_per_sample(w), "profile_ms_per_step": classes,
               "head_kernel_ms_per_step": kern, "head_hbm_bytes": hb, "head_floor_ms_at_copy_peak": floor}
        res["ks"][K] = rec
        print(K, json.dumps(rec), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
