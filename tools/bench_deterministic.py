"""Cost of deterministic mode (gmvae_config::deterministic) against the default mode, measured the way bench.py measures:
graph replay of the whole training step, L2 flushed (256 MB write) between timed steps, CUDA events.  The two modes run in
the same process, alternating, `--repeats` times each; per workload the JSON holds samples/s of both modes per repeat, the
per-class device time of three eager steps, and (torch.profiler, a run of its own) the device time per step of the chained
kernel, the column sums and the reduction step.  Also records whether two default-mode engines drift apart bitwise over 5 steps
of cfg4 -- the reason the mode exists.

    python tools/bench_deterministic.py --out profiles/deterministic/cost.json
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from bench import WORKLOADS, synthetic_images  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def engine(w, det):
    import gmvae_b200
    return gmvae_b200.Engine(model=w["model"], data_size=784, latent_size=w["latent_size"], hidden_sizes=w["hidden_sizes"],
                             mixture_components=w["mixture_components"], max_batch=w["batch"], seed=1234, deterministic=det)


def timed(eng, step, steps, l2, side):
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    with torch.cuda.stream(side):
        for a, b in ev:
            l2.add_(1)
            a.record(side)
            step()
            b.record(side)
    side.synchronize()
    ms = sorted(a.elapsed_time(b) for a, b in ev)
    return ms[len(ms) // 2]


def profile(eng, x, l2, side):
    with torch.cuda.stream(side):
        eng.profile(True)
        for _ in range(3):
            l2.add_(1)
            eng.train_step(x)
        side.synchronize()
        out = {k: v["ms"] / 3 for k, v in eng.profile_read().items()}
        eng.profile(False)
        # per kernel (the reduction step shares profile class bias_grad with the column sums): torch.profiler, a run of its own
        from torch.profiler import ProfilerActivity, profile as tprofile
        with tprofile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(3):
                eng.train_step(x)
            side.synchronize()
        per = {}
        for ev in prof.key_averages():
            for tag in ("gemm_chain_kernel", "det_reduce_kernel", "colsum_kernel"):
                if tag in ev.key:
                    t = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0)   # us
                    per[tag] = per.get(tag, 0.0) + t / 1e3 / 3
        out["kernel_ms_per_step"] = per
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="cfg3,cfg4,cfg5")
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    side = torch.cuda.Stream(dev)
    l2 = torch.zeros(64 * 1024 * 1024, dtype=torch.float32, device=dev)
    res = {"card": card(), "method": "graph replay, L2 flushed between timed steps, CUDA events, median of --steps per repeat; "
           "modes alternate within each repeat", "workloads": {}}
    for name in args.workloads.split(","):
        w = WORKLOADS[name]
        B = w["batch"]
        x = synthetic_images(B, 1234).to(dev)
        engs = {"default": engine(w, False), "deterministic": engine(w, True)}
        steps = {}
        with torch.cuda.stream(side):
            for mode, e in engs.items():
                for _ in range(3):
                    e.train_step(x)
                e.capture_step(x)
                for _ in range(5):
                    e.replay()
                steps[mode] = e.replay
        side.synchronize()
        rep = {m: [] for m in engs}
        for _ in range(args.repeats):
            for m, e in engs.items():
                ms = timed(e, steps[m], args.steps, l2, side)
                rep[m].append({"ms_per_step": ms, "samples_per_s": B / ms * 1e3})
        res["workloads"][name] = {"batch": B, "repeats": rep, "profile_ms_per_step": {m: profile(e, x, l2, side) for m, e in engs.items()}}
        for e in engs.values():
            e.close()
        print(name, json.dumps(res["workloads"][name]), flush=True)
    # one-off record: two default-mode engines, same seed and data, 5 eager steps on the device noise
    w = WORKLOADS["cfg4"]
    x = synthetic_images(w["batch"], 1234).to(dev)
    params = []
    for det in (False, False, True, True):
        e = engine(w, det)
        for _ in range(5):
            e.train_step(x)
        torch.cuda.synchronize()
        params.append(e.params.clone())
        e.close()
    res["cfg4_5_steps_two_engines"] = {
        "default_bitwise_equal": bool(torch.equal(params[0], params[1])),
        "default_params_differing": int((params[0] != params[1]).sum()),
        "default_max_abs_diff": float((params[0] - params[1]).abs().max()),
        "deterministic_bitwise_equal": bool(torch.equal(params[2], params[3])),
        "n_params": params[0].numel()}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["cfg4_5_steps_two_engines"]))


if __name__ == "__main__":
    main()
