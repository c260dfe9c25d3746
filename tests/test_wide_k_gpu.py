"""GMVAE with 128 < K <= 1024 mixture components (objective R): the wide q(y|x) heads (kernels.cuh head_y_wide_*) in the
training step and in every inference entry point, against the fp64 oracle.

The bars are those of tests/test_step_gpu.py (fp32: every loss term and gradient tensor within 1e-5; bf16: terms against the
exact oracle through bf16_term_ok, gradients against the exact oracle and against the bf16 rounding model) and of
tests/test_infer_gpu.py (element-wise, in units of the absolute network).  K covers each register width of the head (256, 512,
1024) on both sides of its boundary: 129 and 256 on the 256-wide kernel, 300 and 500 on the 512-wide one, 1000 and 1024 on
the 1024-wide one."""
import json
import os

import numpy as np
import pytest
import torch

import gmvae_b200
from gmvae_b200 import data, run_gmvae, runners
from oracle import gmvae_oracle as O
from tests import regimes as R
from tests.helpers import Bf16Model, bf16_term_ok, grad_errors, make_engine, make_spec, perturbed_params, rel, run_parity, term_errors
from tests.test_deterministic_gpu import _assert_same, _data, _engine, _run, _state
from tests.test_infer_gpu import compare
from tests.test_step_gpu import GRAD_BF16_EXACT, TOL, _record

pytestmark = pytest.mark.gpu


def small(K, batch=260):
    """The k128 case of tests/test_deterministic_gpu.py at K components: no width a multiple of a tile."""
    return dict(model="gmvae", latent_size=20, hidden_sizes=[90], mixture_components=K, batch=batch, data_size=150)


def cfg3(K, batch=100):
    return dict(model="gmvae", latent_size=64, hidden_sizes=[512, 512], mixture_components=K, batch=batch)


FP32_CASES = {f"small_k{K}": small(K) for K in (129, 256, 500, 1000, 1024)}
FP32_CASES["cfg3_k1024"] = cfg3(1024)


@pytest.mark.parametrize("name", list(FP32_CASES))
def test_parity_fp32(name):
    terr, gerr = run_parity(FP32_CASES[name], "fp32")
    _record("wide_k_" + name, {"precision": "fp32", "terms_rel": terr, "grad_max": max(gerr.values())})
    for k, v in {**terr, **gerr}.items():
        assert v < TOL["fp32"], (name, k, v)


def _inputs(B, K, seed=79):
    g = torch.Generator().manual_seed(seed)
    x = (torch.rand(B, 784, generator=g) < torch.rand(784, generator=g)).to(torch.uint8)
    eps = torch.randn(B, 64, generator=g)
    u = torch.rand(B, K, generator=g).clamp_min(torch.finfo(torch.float32).tiny)
    return x, eps, u


# Against the bf16 rounding model: every tensor < 6e-3 and their rms < 3e-3 as in tests/test_step_gpu.py, except at 1024
# components on 100 rows: decoder linear_0/w measured 9.7e-3 and the rms 3.15e-3, every other tensor within the standard bar
# (NVIDIA B200, power limit 1000 W).  On these weights and inputs one pre-activation of the decoder's second layer lies 7.7e-7 of
# its absolute-network scale from zero (under the rounding model; the closest at K = 256 is 2.7e-6), where fp32 accumulation
# order decides the ReLU, and one flipped unit of one sample weighs ~1/sqrt(B) of the decoder's tensors at 100 rows: the kind
# test_step_gpu.MODEL_TENSOR_BOUND bounds for cfg5_small.  The rounding-model oracle evaluated in fp32 moves the rms by only
# 1.6e-4 (it decides that unit as fp64 does).  The same K on 5 000 and 16 384 rows meets the standard bars.
RMS_BOUND = {"cfg3_k1024_B100": 4.5e-3}
TENSOR_BOUND = {("cfg3_k1024_B100", "decoder_fcnet"): 1.5e-2}


def _check_bf16(cfg, tag):
    """One forward_backward on cfg's model: terms against the exact oracle, every tensor against the exact oracle and against
    the bf16 rounding model (the bars of tests/test_step_gpu.py)."""
    spec = make_spec(cfg)
    params = perturbed_params(spec)
    x, eps, u = _inputs(cfg["batch"], cfg["mixture_components"])
    eng = make_engine(cfg, "bf16")
    eng.set_parameters(params)
    t = eng.forward_backward(x, eps=eps, gumbel_u=u).cpu().tolist()
    out = {}
    for which, q in (("exact", O.EXACT), ("model", Bf16Model(True))):
        terms_ref, grads_ref = O.loss_and_grads(spec, params, x.bool(), eps, u, q=q)
        out[which] = (term_errors(t, terms_ref, spec), grad_errors(eng, grads_ref), {k: terms_ref[k].item() for k in terms_ref if k in
                                                                                      ("loss", "nll", "kl_div_z", "nent")})
    eng.close()
    terr, gerr, ref = out["exact"]
    gerr_model = out["model"][1]
    flat = sum(v * v for v in gerr_model.values()) ** 0.5 / len(gerr_model) ** 0.5
    _record("wide_k_" + tag, {"precision": "bf16", "terms_rel": terr, "terms_ref": ref, "grad_vs_exact_max": max(gerr.values()),
                              "grad_vs_model_max": max(gerr_model.values()), "grad_vs_model_rms": flat})
    bad = bf16_term_ok(terr, ref, TOL["bf16"])
    assert not bad, (tag, "loss terms vs exact oracle (value, limit)", bad)
    assert max(gerr.values()) < GRAD_BF16_EXACT, (tag, gerr)
    assert flat < RMS_BOUND.get(tag, 1.5 * TOL["bf16"]), (tag, flat, gerr_model)
    for k, v in gerr_model.items():
        assert v < TENSOR_BOUND.get((tag, k.split("/")[0]), 3 * TOL["bf16"]), (tag, "vs bf16 rounding model", k, v)


# batch 100: five chained launches with the heads as kernels in between; 5 000: the one-launch plan (from 4 096 rows), the wide
# head between its chained launches; 16 384: cfg4's batch
@pytest.mark.parametrize("K,B", [(256, 100), (1024, 100), (256, 5000), (1024, 5000), (1024, 16384)])
def test_parity_bf16(K, B):
    _check_bf16(cfg3(K, B), f"cfg3_k{K}_B{B}")


def _fp32_gap_bound(spec, params, x, eps, u, terms_ref, grads_ref):
    """Per term / tensor: 1e-5, or twice what the oracle evaluated in fp32 moves it from the fp64 oracle where that is more (the
    rule of tests/test_trained_regime_gpu.py FP32_BOUND: a nearly one-hot softmax loses nent's digits in fp32 arithmetic)."""
    p32 = {k: v.float() for k, v in params.items()}
    t32, g32 = O.loss_and_grads(spec, p32, x, eps, u)
    bound = {}
    for k in ("loss", "nll", "kl_div_z", "nent"):
        bound[k] = max(TOL["fp32"], 2 * rel(t32[k].item(), terms_ref[k].item()))
    for n, g in grads_ref.items():
        bound[n] = max(TOL["fp32"], 2 * ((g32[n].double() - g).norm() / g.norm().clamp_min(1e-30)).item())
    return bound


def test_peaked_y_fp32():
    """q(y|x) nearly one-hot over 1024 components (tests/regimes.py peaked_y: the margin of component 0 is 15.5 + ln 1023 nats
    on the median row), so that the tied-maximum form of the log-sum-exp (lse_above_max) carries the entropy."""
    cfg = small(1024)
    spec = make_spec(cfg)
    params = R.peaked_y(spec, perturbed_params(spec))
    x, _, eps, u = O.synthetic_batch(spec, cfg["batch"])
    terms_ref, grads_ref = O.loss_and_grads(spec, params, x, eps, u)
    bound = _fp32_gap_bound(spec, params, x, eps, u, terms_ref, grads_ref)
    eng = make_engine(cfg, "fp32")
    eng.set_parameters(params)
    t = eng.forward_backward(x, eps=eps, gumbel_u=u).cpu().tolist()
    terr, gerr = term_errors(t, terms_ref, spec), grad_errors(eng, grads_ref)
    eng.close()
    _record("wide_k_peaked_y_k1024", {"precision": "fp32", "terms_rel": terr, "grad": gerr, "bound": bound})
    assert -1e-2 < terms_ref["nent"].item() < 0, terms_ref["nent"]           # the regime holds: q(y|x) nearly one-hot
    for k, v in {**terr, **gerr}.items():
        assert v < bound[k], (k, v, bound[k])


def test_adam_steps_fp32():
    """Three fp32 Adam steps at K = 300 against the oracle's trajectory (as test_step_gpu.test_marginal_training_steps)."""
    cfg = small(300)
    spec = make_spec(cfg)
    params = perturbed_params(spec)
    eng = make_engine(cfg, "fp32", learning_rate=1e-3)
    eng.set_parameters(params)
    st = O.adam_init(params)
    for step in range(3):
        x, _, eps, u = O.synthetic_batch(spec, cfg["batch"], seed_data=100 + step, seed_noise=200 + step)
        terms, _ = O.train_step(spec, params, st, x, eps, u, lr=1e-3)
        loss = eng.train_step(x, eps=eps, gumbel_u=u)
        assert rel(loss[0].item(), terms["loss"].item()) < 1e-5, step
    assert eng.global_step == 3
    for n, v in eng.parameters().items():
        r = params[n]
        assert ((v.cpu().double().reshape(r.shape) - r).norm() / r.norm().clamp_min(1e-30)).item() < 2e-5, n
    eng.close()


# ---------------------------------------------------------------------------------------------------- deterministic mode
DET = small(256)


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_deterministic_two_engines_agree(precision):
    x = _data(DET)
    a, b = _engine(DET, precision), _engine(DET, precision)
    for i, (sa, sb) in enumerate(zip(_run(a, x, 5), _run(b, x, 5))):
        _assert_same(sa, sb, f"step {i}")
    a.close(); b.close()


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_deterministic_matches_default_mode(precision):
    x = _data(DET)
    a, b = _engine(DET, precision, deterministic=False), _engine(DET, precision)
    la, lb = a.forward_backward(x), b.forward_backward(x)
    torch.cuda.synchronize()
    for n, ga in a.gradients().items():
        gb = b.gradients()[n]
        assert ((ga - gb).norm() / ga.norm().clamp_min(1e-30)).item() <= 1e-5, n
    assert torch.allclose(la, lb, rtol=1e-5, atol=0), (la, lb)
    a.close(); b.close()


def test_deterministic_eager_equals_graph():
    x = _data(DET)
    a, b = _engine(DET, "bf16"), _engine(DET, "bf16")
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


# ---------------------------------------------------------------------------------------------------- inference
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_inference_entry_points(precision):
    """encode (logits_y, z_mean, z_sample: what encoder_y_logits / transform / reconstruct_images return), decode and the four
    conditionals, element by element against the oracle's blocks at K = 1024."""
    cfg = small(1024)
    spec = make_spec(cfg)
    params = perturbed_params(spec)
    x, _, eps, u = O.synthetic_batch(spec, cfg["batch"])
    compare("wide_k_small_k1024", precision, spec, params, x, eps, u)


def test_model_class_accessors():
    """The drop-in GMVAE at K = 1024 (fp32 mode): encoder_y(x) (logits and a relaxed sample), prior_gmm(one_hot(k)),
    encoder_y_logits / transform, and generate_samples over the first and the last component."""
    K, Z, D = 1024, 20, 150
    cfg = small(K)
    spec = make_spec(dict(cfg, sigma_min=0.0, raw_sigma_bias=0.5))
    params = perturbed_params(spec)
    x, _, eps, u = O.synthetic_batch(spec, 64)
    m = gmvae_b200.create_gmvae(D, Z, mixture_components=K, fcnet_hidden_sizes=[90], sigma_min=0.0, raw_sigma_bias=0.5, random_seed=7)
    m.configure(precision="fp32", max_batch=128)
    m.engine().set_parameters(params)
    p = {k: v.double() for k, v in params.items()}
    logits_ref = O.mlp(p, "encoder_y", x.double(), 2)

    qy = m.encoder_y(x)
    assert (qy.logits.cpu().double() - logits_ref).abs().max().item() < 1e-4
    y = qy.sample(u=u)
    y_ref = O.gumbel_softmax_sample(qy.logits.cpu().double(), u.double(), 1.0)
    assert tuple(y.shape) == (64, K) and (y.cpu().double() - y_ref).abs().max().item() < 1e-6
    assert (m.encoder_y_logits(x).cpu().double() - logits_ref).abs().max().item() < 1e-4
    assert tuple(m.transform(x).shape) == (64, Z)

    ks = torch.tensor([0, 1, 511, 1023])
    onehot = torch.nn.functional.one_hot(ks, K).float()
    pz = m.prior_gmm(onehot)
    mu_ref, sg_ref = O.normal_params(spec, O.mlp(p, "prior_gmm", onehot.double(), 1))
    assert (pz.mean().cpu().double() - mu_ref).abs().max().item() < 1e-6
    assert (pz.stddev().cpu().double() - sg_ref).abs().max().item() < 1e-6

    s = m.generate_samples(3, clusters=[0, 1023])
    assert tuple(s.shape) == (6, Z)
    eps_s = torch.randn(3, 2, Z, generator=torch.Generator().manual_seed(7)).double()
    mu2, sg2 = O.normal_params(spec, O.mlp(p, "prior_gmm", torch.eye(K, dtype=torch.float64)[[0, 1023]], 1))
    want = (mu2[None] + sg2[None] * eps_s).reshape(6, Z)
    assert (s.cpu().double() - want).abs().max().item() < 1e-5
    m.engine().close()


# ---------------------------------------------------------------------------------------------------- the command line
def test_cli_train_then_eval(tmp_path, monkeypatch):
    monkeypatch.setattr(data, "SPLIT_SIZES", {"train": 2048, "test": 300})       # synthetic stand-in, small
    monkeypatch.delenv("GMVAE_MNIST_DIR", raising=False)

    def flags(*extra):
        return run_gmvae.build_parser().parse_args(
            ["--latent_size=8", "--hidden_size=64", "--num_layers=1", "--batch_size=64", f"--logdir={tmp_path}/logs", "--random_seed=7",
             "--summarise_every=20", "--model=gmvae", "--mixture_components=256"] + list(extra))
    cfg = flags("--mode=train", "--max_steps=39", "--image_summaries=0")
    eng = runners.run_train(cfg)
    assert eng.global_step == 40
    eng.close()
    logdir = runners.logdir_for(cfg)
    recs = [json.loads(l) for l in open(os.path.join(logdir, "summaries.jsonl"))]
    assert [r["step"] for r in recs] == [20, 40]
    assert all("cluster_acc" in r and np.isfinite(list(r.values())).all() for r in recs)
    ck = torch.load(os.path.join(logdir, "model.ckpt-40"))
    assert tuple(ck["encoder_y_fcnet/linear_1/w"].shape) == (64, 256)
    res = runners.run_eval(flags("--mode=eval", "--split=test"), max_wait=0.0)
    assert res["step"] == 40 and res["z"].shape == (300, 8)
    assert np.isfinite(res["z"]).all() and np.isfinite(res["loss_per_example"])
