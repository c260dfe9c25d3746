#!/usr/bin/env python
"""bench.py -- GMVAE training-step throughput (fwd + bwd + Adam) on N B200s of one node.

    python bench.py --gpus 1 --steps 50 --warmup 5
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # the reference's step restated on the host CPU
    python bench.py --dump-outputs DIR ...    # also write the last timed step's results to DIR/<name>.npy

One "step" = one iteration of the reference's hot loop `sess.run([train_op, global_step])`
(/root/reference/scripts/runners.py:231-232) on one synthetic batch.  Rank 0 prints ONE JSON line.
Workload = BASELINE.json configs[3]: GMVAE K=10, z=64, MLP 784-512-512, batch 16384 per GPU,
data-parallel (weak scaling) with an NCCL gradient all-reduce.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# NCCL_DEBUG is left as the caller set it (the driver reads the communicator lines NCCL prints); GMVAE_NCCL_DEBUG overrides.
if os.environ.get("GMVAE_NCCL_DEBUG"):
    os.environ["NCCL_DEBUG"] = os.environ["GMVAE_NCCL_DEBUG"]

import torch  # noqa: E402

WORKLOADS = {
    "cfg4": dict(model="gmvae", latent_size=64, hidden_sizes=[512, 512], mixture_components=10, batch=16384,
                 desc="cfg4 (BASELINE.json configs[3]): GMVAE K=10 z=64 MLP 784-512-512 batch 16384/GPU"),
    "cfg5": dict(model="gmvae", latent_size=128, hidden_sizes=[1024, 1024], mixture_components=50, batch=65536,
                 desc="cfg5 (BASELINE.json configs[4]): GMVAE K=50 z=128 MLP 784-1024-1024 batch 65536/GPU"),
    "cfg3": dict(model="gmvae", latent_size=64, hidden_sizes=[512, 512], mixture_components=10, batch=100,
                 desc="cfg3 (BASELINE.json configs[2]): GMVAE K=10 z=64 MLP 784-512-512 batch 100"),
}
D = 784


def flops_per_sample(w, objective="reference"):
    """2*MACs of forward + weight-gradient + data-gradient GEMMs; the data gradient w.r.t. the
    image is excluded (never needed).  Matches BASELINE.md section 3 (objective R)."""
    H, Z, K = w["hidden_sizes"], w["latent_size"], w["mixture_components"]

    def mlp(i, o):
        sizes = [i] + H + [o]
        return [(sizes[j], sizes[j + 1]) for j in range(len(sizes) - 1)]
    if objective == "marginal":
        # SURVEY.md section 8(a): encoder_y as in R; the x-projection of encoder_gmm layer 0 once per sample
        # (forward + weight gradient, no data gradient); per component: encoder_gmm layers >= 1 and the
        # whole decoder, forward + weight gradient + data gradient.
        ey = mlp(D, K)
        fwd = sum(i * o for i, o in ey) + D * H[0]
        dg = sum(i * o for i, o in ey[1:])
        per = mlp(0, 2 * Z)[1:] + mlp(Z, D)
        fwd += K * sum(i * o for i, o in per)
        dg += K * sum(i * o for i, o in per)
        return 2 * (2 * fwd + dg)
    fwd = dgrad = 0
    nets = [("enc_y", mlp(D, K), False), ("enc_gmm", mlp(D + K, 2 * Z), True), ("prior", [(K, 2 * Z)], True),
            ("dec", mlp(Z, D), True)] if w["model"] == "gmvae" else [("enc", mlp(D, 2 * Z), False), ("dec", mlp(Z, D), True)]
    for name, layers, need_input_grad in nets:
        for j, (i, o) in enumerate(layers):
            fwd += i * o
            if j > 0:
                dgrad += i * o
            elif need_input_grad:
                dgrad += (i - D if name == "enc_gmm" else i) * o   # only the y / z columns need a data gradient
    return 2 * (2 * fwd + dgrad)


def tc_flops_per_sample(w, objective="reference"):
    """FLOPs of the wide contractions (in >= 32 and out >= 32), the ones the roofline fraction is quoted
    on; the thin ones (K or N = mixture components) also run in the tcgen05 kernel but are bandwidth-bound
    and are left out of the numerator (conservative)."""
    if objective == "marginal":
        return flops_per_sample(w, objective) - 2 * 3 * w["hidden_sizes"][-1] * w["mixture_components"]
    H, Z, K = w["hidden_sizes"], w["latent_size"], w["mixture_components"]

    def mlp(i, o):
        sizes = [i] + H + [o]
        return [(sizes[j], sizes[j + 1]) for j in range(len(sizes) - 1)]
    tot = 0
    nets = [("enc_y", mlp(D, K)), ("enc_gmm", mlp(D, 2 * Z)), ("dec", mlp(Z, D))] if w["model"] == "gmvae" else \
           [("enc", mlp(D, 2 * Z)), ("dec", mlp(Z, D))]
    for name, layers in nets:
        for j, (i, o) in enumerate(layers):
            if i >= 32 and o >= 32:
                tot += 2 * i * o + (i * o if (j > 0 or name == "dec") else 0)
    return 2 * tot


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", 1346.3), d.get("hbm_gbs", 6533.2), "MEASURED_PEAKS.json bf16_tflops_sustained"
    return 1400.0, 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def wait_first(self, timeout=3.0):
        t0 = time.time()
        while self.proc is not None and not self.rows and time.time() - t0 < timeout:
            time.sleep(0.01)

    def mark(self):
        """Call at the start of the timed region."""
        self.begin = len(self.rows)

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        rows_all = self.rows
        self.rows = rows_all[getattr(self, "begin", 0):] or rows_all[-3:]     # a sub-100 ms region may see no tick of its own
        sm = sorted(int(float(r[1])) for r in self.rows if len(r) >= 8 and r[1].replace(".", "").isdigit())
        mx = [int(float(r[2])) for r in self.rows if len(r) >= 8 and r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 8 for n, v in zip(names, r[4:8]) if v.lower().startswith("active")})
        pw = [float(r[3]) for r in self.rows if len(r) >= 8 and r[3].replace(".", "").isdigit()]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm), "power_w_max": max(pw) if pw else None}


def synthetic_images(batch, seed):
    """SURVEY.md section 8(d): per-pixel rate p_d ~ U(0,1) drawn once; x = U(0,1) < p_d (bool)."""
    g = torch.Generator().manual_seed(seed)
    p = torch.rand(D, generator=g)
    return (torch.rand(batch, D, generator=g) < p).to(torch.uint8)


# ------------------------------------------------------------------------------------ CPU arm
def cpu_step_rate(w, sample_batch, steps, threads):
    """The reference's training step restated on the CPU (oracle/, PyTorch fp32, autograd backward,
    TF-form Adam) -- `kind: "port"`: TF 1.13 cannot be installed here (SURVEY.md F3)."""
    from oracle import gmvae_oracle as O
    torch.set_num_threads(threads)
    spec = O.Spec(w["model"], D, w["latent_size"], list(w["hidden_sizes"]), w["mixture_components"])
    params = O.init_params(spec, dtype=torch.float32)
    st = O.adam_init(params)
    x, _, eps, u = O.synthetic_batch(spec, sample_batch)
    O.train_step(spec, params, st, x, eps, u)       # warm-up
    t0 = time.perf_counter()
    for _ in range(steps):
        O.train_step(spec, params, st, x, eps, u)
    dt = time.perf_counter() - t0
    return sample_batch * steps / dt, dt


def run_reference_arm(args, w):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    sample = min(w["batch"], 4096)
    for _ in range(max(args.warmup, 1) - 1):
        cpu_step_rate(w, sample, 1, cores)
    _, dt1 = cpu_step_rate(w, sample, 2, cores)
    # bounded: at most args.steps steps and at most ~60 s of CPU work
    nsteps = max(1, min(args.steps, int(60.0 / max(dt1 / 2, 1e-4))))
    rate, dt = cpu_step_rate(w, sample, nsteps, cores)
    args.steps = nsteps
    # the reference's own session config pins TF to one intra-op and one inter-op thread (runners.py:203-204):
    # the same step on ONE thread, a bounded sample, reported beside the all-cores number
    one_steps = max(1, min(3, int(10.0 / max(dt / max(nsteps, 1) * cores * 0.5, 1e-3))))
    rate1, dt1t = cpu_step_rate(w, sample, one_steps, 1)
    line = {
        "impl": "reference", "metric": "GMVAE train samples/sec (fwd+bwd+Adam)", "value": rate, "unit": "samples/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / max(args.steps, 1),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": w["desc"], "objective": "reference (gmvae.py:238-267)", "note": "host CPU only; GPUs idle"},
        "cpu_baseline": {"value": rate, "unit": "samples/s", "cores": cores, "kind": "port",
                         "sample": f"{sample} samples/step x {args.steps} steps of the same model (restated reference graph on "
                                   f"PyTorch-CPU fp32; TF 1.13 not installable)"},
        "cpu_baseline_single_thread": {"value": rate1, "unit": "samples/s", "cores": 1, "kind": "port",
                                       "sample": f"{sample} samples/step x {one_steps} steps ({dt1t:.1f} s); the reference's own "
                                                 f"ConfigProto uses intra_op = inter_op = 1 (runners.py:203-204)"},
        "e2e": {"value": rate, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------ GPU arm
def flush_l2(buf):
    buf.add_(1)


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(eng, out_dir):
    """What a caller of the timed step receives from it: the loss terms [loss, nll, kl_div_z, nent] and every parameter as
    Adam left it, float32, one DIR/<name>.npy each ("/" in a variable name becomes ".").  The step they come from starts from
    the engine's seeded initial state (run_gpu_arm restores it, untimed, before the last timed step) on the seeded batch, with
    noise keyed by seed and step: the batch is reduce-added across CTAs in no fixed order, so steps that build on earlier
    ones would carry that rounding forward, amplified by Adam.  Two runs, or two builds, with the same arguments can
    therefore be compared array for array."""
    import numpy as np
    arrays = {"loss_terms": eng.loss_buf}
    arrays.update(("param." + name.replace("/", "."), v) for name, v in eng.parameters().items())
    arrays = {k: v.detach().float().cpu().numpy() for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes of outputs exceed the {DUMP_LIMIT_BYTES} byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def run_gpu_arm(args, w):
    import torch.distributed as dist
    import gmvae_b200
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a GPU (there is no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B = args.batch or w["batch"]
    eng = gmvae_b200.Engine(model=w["model"], data_size=D, latent_size=w["latent_size"], hidden_sizes=w["hidden_sizes"],
                            mixture_components=w["mixture_components"], precision=args.precision, objective=args.objective,
                            max_batch=B, device=local, seed=1234)   # same weights on every rank; noise is keyed by rank
    if world > 1:
        eng.init_data_parallel()
    init_state = eng.state_dict() if args.dump_outputs else None

    x_host = synthetic_images(B, 1234 + rank).pin_memory()
    x_dev = x_host.to(dev)
    side = torch.cuda.Stream(dev)
    l2_buf = torch.zeros(64 * 1024 * 1024, dtype=torch.float32, device=dev)   # 256 MB > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---- device-resident throughput: graph replay of the whole step ----------------------------
    with torch.cuda.stream(side):
        for _ in range(2):
            eng.train_step(x_dev)
        if args.no_graph:
            step = lambda: eng.train_step(x_dev)
        else:
            eng.capture_step(x_dev)
            step = eng.replay
        for _ in range(args.warmup):
            step()
        side.synchronize()
        n0 = eng.launch_count()
        eng.train_step(x_dev)
        launches_per_step = eng.launch_count() - n0
        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()
            sampler.wait_first()
        for _ in range(3):
            step()                                # keep the GPU under load until the sampler ticks
        barrier()
        # Device-side rendezvous: the ranks leave the host barrier a few hundred microseconds to milliseconds apart; two
        # untimed steps (each ends in the gradient all-reduce, which no rank leaves before every rank has entered it) line
        # the streams up, so the first timed event does not contain the start skew.
        for _ in range(2 if world > 1 else 0):
            flush_l2(l2_buf)
            step()
        if rank == 0:
            sampler.mark()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        for i in range(args.steps):
            if init_state is not None and i == args.steps - 1:
                eng.load_state_dict(init_state)   # the dumped step starts from the seeded initial state (untimed)
            flush_l2(l2_buf)                      # evict the previous step's tensors from L2 (untimed)
            ev[i][0].record(side)
            step()
            ev[i][1].record(side)
        barrier()
        clocks = sampler.stop() if rank == 0 else None
        step_ms = sorted(a.elapsed_time(b) for a, b in ev)
        dev_ms = sum(step_ms)
        med_ms = step_ms[len(step_ms) // 2]
        loss_terms = eng.loss_buf.cpu().tolist()
        if args.dump_outputs and rank == 0:
            dump_outputs(eng, args.dump_outputs)

        # ---- per-kernel-class device time: CUDA events after every launch of 3 eager steps --------
        prof_steps = 3
        eng.profile(True)
        for _ in range(prof_steps):
            flush_l2(l2_buf)
            eng.train_step(x_dev)
        side.synchronize()
        prof = {k: {"ms_per_step": v["ms"] / prof_steps, "launches_per_step": v["launches"] // prof_steps}
                for k, v in eng.profile_read().items()}
        eng.profile(False)

        # ---- input pipeline kernel (SURVEY 8 row f3): dynamic binarisation of one batch of device-resident intensities ----
        inten = torch.randint(0, 256, (B, D), dtype=torch.uint8, device=dev)
        x_bin = torch.empty_like(x_dev)
        for i in range(3):
            eng.binarize(inten, out=x_bin, draw=i)
        evb = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(20)]
        for i, (a, b) in enumerate(evb):
            flush_l2(l2_buf)
            a.record(side)
            eng.binarize(inten, out=x_bin, draw=3 + i)
            b.record(side)
        side.synchronize()
        bin_ms = sorted(a.elapsed_time(b) for a, b in evb)[len(evb) // 2]
        del inten, x_bin

        # ---- end to end: pinned host batch -> H2D -> step -> D2H loss, every step ----------------
        # The host batch is the binary image 1 bit per pixel (numpy.packbits order, 98 bytes per image): what the input of
        # this path is (runners.py:44-47 feeds {0,1}); Engine.unpack_bits expands it on the device into the captured step's
        # input buffer.  H2D bytes per step = B * 98.
        import numpy as np
        packed_host = torch.from_numpy(np.packbits(x_host.numpy(), axis=1)).pin_memory()
        copy_stream = torch.cuda.Stream(dev)
        stage = [torch.empty(packed_host.shape, dtype=torch.uint8, device=dev) for _ in range(2)]
        ready = [torch.cuda.Event() for _ in range(2)]
        consumed = [torch.cuda.Event() for _ in range(2)]
        loss_host = torch.zeros(args.steps + args.warmup + 2, 4).pin_memory()

        def e2e_loop(n, off):
            for i in range(n):
                s = i % 2
                with torch.cuda.stream(copy_stream):
                    copy_stream.wait_event(consumed[s])
                    stage[s].copy_(packed_host, non_blocking=True)
                    ready[s].record(copy_stream)
                side.wait_event(ready[s])
                eng.unpack_bits(stage[s], out=x_dev)
                consumed[s].record(side)
                step()
                loss_host[off + i].copy_(eng.loss_buf, non_blocking=True)
        for s in range(2):
            consumed[s].record(side)
        e2e_loop(args.warmup, 0)
        barrier()
        if world > 1:
            e2e_loop(2, args.warmup)              # device-side rendezvous, as above
        t0 = torch.cuda.Event(enable_timing=True); t1 = torch.cuda.Event(enable_timing=True)
        t0.record(side)
        e2e_loop(args.steps, args.warmup + 2)
        t1.record(side)
        barrier()
        e2e_ms = t0.elapsed_time(t1)
        assert torch.equal(x_dev.cpu(), x_host), "unpacked batch differs from the host batch"
        h2d_bytes = int(packed_host.numel())

    # max over ranks
    if world > 1:
        t = torch.tensor([dev_ms, e2e_ms, med_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_ms, e2e_ms, med_ms = t.tolist()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peak_tf, peak_hbm, peak_src = measured_peaks()
    # DRAM traffic of the dominant kernel from the committed `ncu --set full` capture (profiles/), per launch
    traffic = None
    tp = os.path.join(ROOT, "profiles", "r2_traffic.json")
    if os.path.exists(tp):
        tj = json.load(open(tp)).get(f"{args.workload}:{args.objective}:{args.precision}")
        if tj and world == 1 and B == w["batch"]:
            traffic = tj["dram_bytes_tc_gemm_per_step"] / max(tj["tc_launches_per_step"], 1)
    fps = flops_per_sample(w, args.objective)
    # `value` is the mean over EXACTLY args.steps timed steps (max over ranks); the median per-step time is reported beside it
    # (a one-off stall -- clock ramp, a late rank -- moves the mean of a 20-step run, not the median)
    ms_per_step = dev_ms / args.steps
    value = world * B * args.steps / (dev_ms * 1e-3)
    step_tf = (B * fps) / (ms_per_step * 1e-3) / 1e12
    tc_ms = prof["tc_gemm_fwd_dgrad"]["ms_per_step"] + prof["tc_gemm_wgrad"]["ms_per_step"]
    tc_launches = prof["tc_gemm_fwd_dgrad"]["launches_per_step"] + prof["tc_gemm_wgrad"]["launches_per_step"]
    achieved_tf = (B * tc_flops_per_sample(w, args.objective)) / (tc_ms * 1e-3) / 1e12 if tc_ms > 0 else 0.0
    e2e_value = world * B * args.steps / (e2e_ms * 1e-3)
    line = {
        "metric": "GMVAE train samples/sec (fwd+bwd+Adam)", "value": value, "unit": "samples/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "ms_per_step_median": med_ms,
        "ms_per_step_max": step_ms[-1], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": args.precision, "data": "synthetic",
        "config": {"workload": w["desc"], "objective": args.objective, "global_batch": world * B, "parallelism": f"dp{world}",
                   "l2": "L2 flushed (256 MB write) between timed steps", "graph": not args.no_graph,
                   "noise": "drawn on device (Philox) each step", "loss_terms": loss_terms},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "samples/s", "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 16,
                "ms_per_step": e2e_ms / args.steps,
                "note": "pinned bit-packed batch (98 B/image) -> H2D (copy stream, double-buffered) -> unpack on device -> graph -> D2H loss"},
        "gpu_launches": int(launches_per_step * args.steps),
        "roofline": {"bound": "tensor", "achieved": achieved_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved_tf / peak_tf,
                     "traffic": traffic, "kernel": f"gemm_chain_kernel (tcgen05 GEMM jobs + fused epilogues/heads; {tc_launches} launches/step, {tc_ms:.3f} ms/step by CUDA events)",
                     "peak_source": peak_src, "flop_per_sample": fps, "tc_flop_per_sample": tc_flops_per_sample(w, args.objective),
                     "whole_step_tflops": step_tf, "whole_step_frac": step_tf / peak_tf},
        "kernel_profile": prof,
        "comm_exposed_ms": prof.get("comm", {}).get("ms_per_step", 0.0),
        "input_pipeline": {"kernel": "binarize_kernel (runners.py:44-47 on device-resident intensities; not part of the timed step)",
                           "bound": "hbm", "achieved": 2.0 * B * D / (bin_ms * 1e-3) / 1e9, "peak": peak_hbm, "unit": "GB/s",
                           "frac": 2.0 * B * D / (bin_ms * 1e-3) / 1e9 / peak_hbm, "ms_per_batch": bin_ms,
                           "samples_per_s": B / (bin_ms * 1e-3), "bytes_per_sample": 2 * D},
    }
    if not args.no_cpu_baseline and world == 1:
        cores = os.cpu_count() or 1
        sample = min(B, 4096)
        _, dt1 = cpu_step_rate(w, sample, 2, cores)
        n = max(3, min(2000, int(12.0 / max(dt1 / 2, 1e-4))))         # ~12 s of CPU work
        rate, dt = cpu_step_rate(w, sample, n, cores)
        line["cpu_baseline"] = {"value": rate, "unit": "samples/s", "cores": cores, "kind": "port",
                                "sample": f"{sample} samples/step x {n} steps, restated reference graph on PyTorch-CPU fp32 ({dt:.1f} s)"}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=400)
    ap.add_argument("--warmup", type=int, default=20)      # SURVEY 8(d): >= 20 warm-up launches, >= 200 timed
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg4", choices=list(WORKLOADS))
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--objective", default="reference", choices=["reference", "marginal"])
    ap.add_argument("--batch", type=int, default=0, help="override the per-GPU batch")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's loss terms and parameters to DIR")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU arm (--impl ours)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    w = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference_arm(args, w)
    else:
        run_gpu_arm(args, w)


if __name__ == "__main__":
    main()
