"""bench.py's accounting, checked on the CPU: the algorithmic FLOP counts behind `roofline.achieved` are SURVEY section 8(a)'s
table, the roofline denominators come from MEASURED_PEAKS.json, and the CPU arm prints the contract's JSON line."""
import importlib.util
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    spec = importlib.util.spec_from_file_location("bench_module", os.path.join(ROOT, "bench.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def test_flop_counts_match_survey_table():
    b = _bench()
    cfg4, cfg5, cfg3 = b.WORKLOADS["cfg4"], b.WORKLOADS["cfg5"], b.WORKLOADS["cfg3"]
    assert b.flops_per_sample(cfg4) == 10_997_248 == b.flops_per_sample(cfg3)         # GMVAE (R), K=10 z=64 784-512-512
    assert b.flops_per_sample(cfg5) == 33_164_288                                     # GMVAE (R), K=50 z=128 784-1024-1024
    assert b.flops_per_sample(cfg4, "marginal") == 66_254_848                         # shared x-projection
    assert b.flops_per_sample(cfg5, "marginal") == 1_000_976_384
    vae = dict(model="vae", latent_size=64, hidden_sizes=[512, 512], mixture_components=1)
    assert b.flops_per_sample(vae) == 7_749_632                                       # cfg1 / cfg2
    # the roofline numerator leaves the thin (K-wide) contractions out: never more than the whole
    for w, obj in ((cfg4, "reference"), (cfg5, "reference"), (cfg4, "marginal")):
        assert 0.9 * b.flops_per_sample(w, obj) < b.tc_flops_per_sample(w, obj) <= b.flops_per_sample(w, obj)
    assert b.tc_flops_per_sample(cfg4) == 10_928_128


def test_peaks_come_from_measured_file():
    b = _bench()
    tf, hbm, src = b.measured_peaks()
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        assert tf == d["bf16_tflops_sustained"] and hbm == d["hbm_gbs"] and "MEASURED_PEAKS" in src
    else:
        assert "fallback" in src


def test_reference_arm_prints_the_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "cfg3", "--steps", "2",
                        "--warmup", "1"], capture_output=True, text=True, timeout=300,
                       env=dict(os.environ, RANK="0", WORLD_SIZE="1"))
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "samples/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0 and "cfg3" in d["config"]["workload"]
    one = d["cpu_baseline_single_thread"]                        # the reference pins TF to one thread (runners.py:203-204)
    assert one["cores"] == 1 and one["value"] > 0 and one["kind"] == "port"
    # the other ranks of a torchrun launch exit 0 without work and without output
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1"],
                       capture_output=True, text=True, timeout=120, env=dict(os.environ, RANK="1", WORLD_SIZE="2"))
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_rejected_arguments(tmp_path):
    for extra, msg in ((["--steps", "0"], "--steps must be at least 1"),
                       (["--impl", "reference", "--dump-outputs", str(tmp_path / "d")], "--dump-outputs applies to the GPU arm")):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, capture_output=True, text=True, timeout=120)
        assert r.returncode == 2 and msg in r.stderr and r.stdout == "", (extra, r.stderr[-2000:])
    assert not (tmp_path / "d").exists()
