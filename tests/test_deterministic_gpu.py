"""Deterministic mode on the GPU: two engines with the same seed give bit-identical steps (torch.equal), re-initialising
reproduces a run, graph replay equals eager steps, and the parity bars against the oracle still hold."""
import json
import os
import subprocess
import sys

import pytest
import torch

import gmvae_b200
from oracle import gmvae_oracle as O
from tests.helpers import CONFIGS, Bf16Model, bf16_term_ok, grad_errors, make_engine, make_spec, perturbed_params, term_errors
from tests.test_step_gpu import GRAD_BF16_EXACT, MODEL_TENSOR_BOUND, TOL

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu

CASES = {
    "vae": dict(model="vae", latent_size=64, hidden_sizes=[512, 512], mixture_components=1, batch=100),
    "vae_gmp": dict(model="vae_gmp", latent_size=64, hidden_sizes=[512, 512], mixture_components=10, batch=100),
    "gmvae": dict(model="gmvae", latent_size=64, hidden_sizes=[512, 512], mixture_components=10, batch=100),
    "gmvae_5000": dict(model="gmvae", latent_size=64, hidden_sizes=[512, 512], mixture_components=10, batch=5000),
    "cfg4": dict(model="gmvae", latent_size=64, hidden_sizes=[512, 512], mixture_components=10, batch=16384),
    "cfg5_model": dict(model="gmvae", latent_size=128, hidden_sizes=[1024, 1024], mixture_components=50, batch=8192),
    "k17": dict(model="gmvae", latent_size=40, hidden_sizes=[96, 72], mixture_components=17, batch=150, data_size=200),
}
PARAMS = [(n, "bf16") for n in CASES] + [(n, "fp32") for n in ("vae", "vae_gmp", "gmvae")]


def _engine(cfg, precision, seed=7, deterministic=True):
    return gmvae_b200.Engine(model=cfg["model"], data_size=cfg.get("data_size", 784), latent_size=cfg["latent_size"],
                             hidden_sizes=cfg["hidden_sizes"], mixture_components=cfg["mixture_components"], precision=precision,
                             max_batch=cfg["batch"], seed=seed, deterministic=deterministic)


def _data(cfg, seed=11):
    g = torch.Generator().manual_seed(seed)
    return (torch.rand(cfg["batch"], cfg.get("data_size", 784), generator=g) < 0.3).to(torch.uint8).cuda()


def _state(e, loss):
    torch.cuda.synchronize()
    return {"params": e.params.clone(), "adam_m": e.adam_m.clone(), "adam_v": e.adam_v.clone(), "loss": loss.clone(),
            "step": e.global_step}


def _assert_same(a, b, what):
    for k in a:
        same = a[k] == b[k] if k == "step" else torch.equal(a[k], b[k])
        assert same, (what, k)


def _run(e, x, steps):
    out = []
    for _ in range(steps):
        out.append(_state(e, e.train_step(x)))
    return out


@pytest.mark.parametrize("name,precision", PARAMS)
def test_two_engines_agree(name, precision):
    cfg = CASES[name]
    x = _data(cfg)
    a, b = _engine(cfg, precision), _engine(cfg, precision)
    a.forward_backward(x); b.forward_backward(x)
    torch.cuda.synchronize()
    assert torch.equal(a.grads, b.grads), "gradient buffer"
    assert torch.equal(a.loss_buf, b.loss_buf)
    a.set_global_step(0); b.set_global_step(0)
    for i, (sa, sb) in enumerate(zip(_run(a, x, 5), _run(b, x, 5))):
        _assert_same(sa, sb, f"step {i}")
    a.close(); b.close()


def test_reinitialise_reproduces_the_run():
    cfg = CASES["gmvae"]
    x = _data(cfg)
    e = _engine(cfg, "bf16")
    first = _run(e, x, 5)
    e.initialize(7)
    e.set_global_step(0)
    for i, (s0, s1) in enumerate(zip(first, _run(e, x, 5))):
        _assert_same(s0, s1, f"step {i}")
    e.close()


@pytest.mark.parametrize("name", ["gmvae", "gmvae_5000"])
def test_eager_equals_graph(name):
    cfg = CASES[name]
    x = _data(cfg)
    a, b = _engine(cfg, "bf16"), _engine(cfg, "bf16")
    eager = _run(a, x, 5)
    side = torch.cuda.Stream(b.device)
    with torch.cuda.stream(side):
        b.capture_step(x)
    graph = []
    with torch.cuda.stream(side):
        for _ in range(5):
            graph.append(_state(b, b.replay()))
    for i, (s0, s1) in enumerate(zip(eager, graph)):
        _assert_same(s0, s1, f"step {i}")
    a.close(); b.close()


@pytest.mark.parametrize("name", ["tiny_gmvae", "tiny_vae", "tiny_gmp", "cfg3", "k20_ragged"])
def test_parity_fp32(name):
    cfg = CONFIGS[name]
    spec = make_spec(cfg)
    params = perturbed_params(spec)
    x, _, eps, u = O.synthetic_batch(spec, cfg["batch"])
    terms_ref, grads_ref = O.loss_and_grads(spec, params, x, eps, u)
    eng = make_engine(cfg, "fp32", deterministic=True)
    eng.set_parameters(params)
    t = eng.forward_backward(x, eps=eps, gumbel_u=u).detach().cpu().tolist()
    terr, gerr = term_errors(t, terms_ref, spec), grad_errors(eng, grads_ref)
    eng.close()
    assert max(terr.values()) < 1e-5, terr
    assert max(gerr.values()) < 1e-5, gerr


@pytest.mark.parametrize("name", ["cfg1", "cfg2", "cfg3", "cfg5_small", "k20_ragged"])
def test_parity_bf16(name):
    # the bars of tests/test_step_gpu.py: terms against the exact oracle, gradients against the exact oracle and against the
    # bf16 rounding model
    cfg = CONFIGS[name]
    spec = make_spec(cfg)
    params = perturbed_params(spec)
    x, _, eps, u = O.synthetic_batch(spec, cfg["batch"])
    terms_ref, grads_ref = O.loss_and_grads(spec, params, x, eps, u)
    _, grads_q = O.loss_and_grads(spec, params, x, eps, u, q=Bf16Model(True))
    eng = make_engine(cfg, "bf16", deterministic=True)
    eng.set_parameters(params)
    t = eng.forward_backward(x, eps=eps, gumbel_u=u).detach().cpu().tolist()
    terr, gerr, gerr_model = term_errors(t, terms_ref, spec), grad_errors(eng, grads_ref), grad_errors(eng, grads_q)
    eng.close()
    assert not bf16_term_ok(terr, {k: terms_ref[k].item() for k in terr}, TOL["bf16"]), terr
    assert max(gerr.values()) < GRAD_BF16_EXACT, gerr
    flat = sum(v * v for v in gerr_model.values()) ** 0.5 / len(gerr_model) ** 0.5
    assert flat < 1.5 * TOL["bf16"], flat
    for k, v in gerr_model.items():
        assert v < MODEL_TENSOR_BOUND.get(name, 3 * TOL["bf16"]), (k, v)


@pytest.mark.parametrize("name,precision", [("gmvae", "bf16"), ("vae_gmp", "bf16"), ("gmvae", "fp32"), ("gmvae_5000", "bf16"),
                                            ("cfg4", "bf16"), ("cfg5_model", "bf16")])
def test_matches_default_mode(name, precision):
    # one step of each mode on the same weights, data and noise: the same k-split partials and column sums, added in another order
    cfg = CASES[name]
    x = _data(cfg)
    a, b = _engine(cfg, precision, deterministic=False), _engine(cfg, precision)
    la, lb = a.forward_backward(x), b.forward_backward(x)
    torch.cuda.synchronize()
    for n, ga in a.gradients().items():
        gb = b.gradients()[n]
        assert ((ga - gb).norm() / ga.norm().clamp_min(1e-30)).item() <= 1e-5, n
    assert torch.allclose(la, lb, rtol=1e-5, atol=0), (la, lb)
    a.close(); b.close()


def test_cli_reproduces_a_run(tmp_path):
    def run(d):
        r = subprocess.run([sys.executable, "-m", "gmvae_b200.run_gmvae", "--mode=train", "--model=gmvae", "--deterministic",
                            "--random_seed=7", "--batch_size=4096", "--max_steps=20", "--summarise_every=10", f"--logdir={d}",
                            "--image_summaries=0"], capture_output=True, text=True, timeout=900, cwd=ROOT)
        assert r.returncode == 0, r.stderr[-3000:]
        return d
    a, b = run(tmp_path / "a"), run(tmp_path / "b")
    files = lambda d: sorted(str(p.relative_to(d)) for p in d.rglob("*") if p.is_file())
    assert files(a) == files(b)
    ckpts = [f for f in files(a) if os.path.basename(f).startswith("model.ckpt-")]
    assert ckpts
    for f in ckpts:
        sa, sb = torch.load(a / f, map_location="cpu"), torch.load(b / f, map_location="cpu")
        flat = lambda s: {k: v for k, v in (s.items() if isinstance(s, dict) else []) if torch.is_tensor(v)}
        assert flat(sa).keys() == flat(sb).keys()
        for k in flat(sa):
            assert torch.equal(flat(sa)[k], flat(sb)[k]), (f, k)
    for f in (f for f in files(a) if f.endswith("summaries.jsonl")):
        ra = [json.loads(l) for l in open(a / f)]
        rb = [json.loads(l) for l in open(b / f)]
        strip = lambda r: {k: v for k, v in r.items() if "sec" not in k and "time" not in k}
        assert [strip(r) for r in ra] == [strip(r) for r in rb]


def test_non_finite_stays_non_finite():
    # the fixed-point loss sums flag a NaN addend: the term comes out NaN, as in the default mode, not as a saturated number
    cfg = CASES["gmvae"]
    x = _data(cfg)
    for det in (False, True):
        e = _engine(cfg, "bf16", deterministic=det)
        e.parameters()["decoder_fcnet/linear_2/b"].fill_(float("nan"))
        e.params_updated()
        t = e.forward_backward(x).cpu()
        assert torch.isnan(t[0]) and torch.isnan(t[1]), (det, t)
        e.close()
