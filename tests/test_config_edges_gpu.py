"""The training step away from its default configuration, against the fp64 oracle with the same hyperparameters: the relaxation
temperature, gen_bias_init, the sigma_min clamp (the drop-in defaults and a clamp that is active on about half of the scales),
Adam's hyperparameters and a global step set from outside; then a workspace that holds NaN bytes before the first step and a
handle whose shared buffers were last written by the inference entry points.

Bars are those of tests/test_step_gpu.py: fp32 within 1e-5 of the oracle, bf16 against the exact oracle and the bf16 rounding
model.  tests/test_oracle.py checks that every knob value used here moves the oracle by far more than these bars, so a kernel
that ignored a knob would fail."""
import ctypes as C

import pytest
import torch

from gmvae_b200 import _lib
from oracle import gmvae_oracle as O
from tests.helpers import CONFIGS, active_clamp, clamp_stats, make_engine, make_spec, perturbed_params, rel, run_parity
from tests.test_step_gpu import FULL, TOL, _check_at, _check_bf16, _full_inputs, _record

pytestmark = pytest.mark.gpu

GEN_BIAS = -1.5
DROPIN_SIGMA = dict(sigma_min=0.001, raw_sigma_bias=0.25)     # what create_gmvae / create_vae default to


def _fp32(name, cfg, objective="reference", tag=""):
    terr, gerr = run_parity(cfg, "fp32", objective=objective)
    _record(name, {"precision": "fp32", "objective": objective, "plan": tag, "terms_rel": terr, "grad_max": max(gerr.values())})
    for k, v in {**terr, **gerr}.items():
        assert v < TOL["fp32"], (name, tag, k, v)


def _both(name, cfg, precision, objective="reference", tag="", monkeypatch=None):
    if precision == "fp32":
        _fp32(name, cfg, objective, tag)
    else:
        if objective == "marginal":
            monkeypatch.setenv("GMVAE_M_CHUNK_ROWS", "512")          # as test_parity_marginal_bf16
        _check_bf16(name, objective=objective, tag=tag, cfg=cfg)


# ------------------------------------------------------------------ temperature
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("T", [0.5, 2.0])
@pytest.mark.parametrize("name", ["cfg3", "k20_ragged"])        # y head fused into the GEMM epilogue (K <= 16) / the warp head
def test_temperature(name, T, precision):
    _both(name, dict(CONFIGS[name], temperature=T), precision, tag=f"T={T}")


@pytest.mark.parametrize("T", [0.5, 2.0])
def test_temperature_row_jobs(T):
    # 5 000 rows: the y head runs as a row job of the chained kernel
    _check_at(dict(FULL, temperature=T), 5000, "cfg4_B5000", f"T={T}")


# ------------------------------------------------------------------ gen_bias_init
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("name,objective", [("cfg1", "reference"), ("tiny_gmp", "reference"), ("cfg3", "reference"),
                                            ("tiny_gmvae", "marginal")])
def test_gen_bias_init(name, objective, precision, monkeypatch):
    _both(name, dict(CONFIGS[name], gen_bias_init=GEN_BIAS), precision, objective, f"gen_bias_init={GEN_BIAS}", monkeypatch)


def test_gen_bias_init_row_jobs():
    _check_at(dict(FULL, gen_bias_init=GEN_BIAS), 5000, "cfg4_B5000", f"gen_bias_init={GEN_BIAS}")


def _condition(eng, which, in1, in2, n, width_a, width_b=0):
    """gmvae_condition on device copies of the inputs: (out_a, out_b or None)."""
    in1 = torch.as_tensor(in1).to(eng.device, torch.float32).contiguous()
    in2 = None if in2 is None else torch.as_tensor(in2).to(eng.device, torch.float32).contiguous()
    a = torch.empty(n, width_a, dtype=torch.float32, device=eng.device)
    b = torch.empty(n, width_b, dtype=torch.float32, device=eng.device) if width_b else None
    _lib.check(eng.lib.gmvae_condition(eng._h, which, in1.data_ptr(), None if in2 is None else in2.data_ptr(), n, a.data_ptr(),
                                       None if b is None else b.data_ptr(), eng._stream()), "gmvae_condition")
    return a, b


def _close(a, b, tol):
    b = b.to(torch.float64)
    return ((a.detach().cpu().double() - b).abs().max() / b.abs().max().clamp_min(1e-30)).item() < tol


@pytest.mark.parametrize("precision,tol", [("fp32", 1e-5), ("bf16", 2e-2)])
@pytest.mark.parametrize("name", ["cfg1", "cfg3", "h33_7"])
def test_gen_bias_init_decode(name, precision, tol):
    """decode() = sigmoid(decoder(z) + gen_bias_init) and condition(DECODER) = decoder(z) + gen_bias_init (base.py:130-146)."""
    cfg = dict(CONFIGS[name], gen_bias_init=GEN_BIAS)
    spec = make_spec(cfg)
    params = perturbed_params(spec)
    eng = make_engine(cfg, precision)
    eng.set_parameters(params)
    n = cfg["batch"]
    z = torch.randn(n, spec.latent_size, generator=torch.Generator().manual_seed(5))
    logits_ref = O.mlp(params, "decoder", z.double(), len(spec.hidden_sizes) + 1) + GEN_BIAS
    assert _close(eng.decode(z), torch.sigmoid(logits_ref), tol)
    logits, _ = _condition(eng, 0, z, None, n, spec.data_size)
    assert _close(logits, logits_ref, tol)
    eng.close()


# ------------------------------------------------------------------ sigma_min / raw_sigma_bias
SIGMA_CASES = [("cfg1", "reference"), ("cfg2", "reference"), ("cfg3", "reference"), ("tiny_gmvae", "marginal")]


def _sigma_cfg(name, cfg, knobs, objective, inputs):
    """The drop-in defaults, or an active clamp chosen on the oracle's own scales; the clamped share is recorded and, for the
    active clamp, held to 20-80 % of the scales of q(z) and (GMVAE) of p(z|y), so that the case cannot turn vacuous."""
    params, x, eps, u = inputs
    cfg = dict(cfg, **DROPIN_SIGMA) if knobs == "dropin" else active_clamp(cfg, params, x, eps, u, objective)
    st = clamp_stats(cfg, params, x, eps, u, objective)
    _record(name, {"knobs": knobs, "objective": objective, "clamp": st})
    if knobs == "active":
        for k in ("sigma_q_clamped", "sigma_p_clamped"):
            if k in st:
                assert 0.2 <= st[k] <= 0.8, (name, k, st)
    return cfg


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("knobs", ["dropin", "active"])
@pytest.mark.parametrize("name,objective", SIGMA_CASES)
def test_sigma_min(name, objective, knobs, precision, monkeypatch):
    cfg = CONFIGS[name]
    spec = make_spec(cfg)
    x, _, eps, u = O.synthetic_batch(spec, cfg["batch"], objective=objective)
    cfg = _sigma_cfg(name, cfg, knobs, objective, (perturbed_params(spec), x, eps, u))
    _both(name, cfg, precision, objective, f"sigma={knobs}", monkeypatch)


@pytest.mark.parametrize("knobs", ["dropin", "active"])
def test_sigma_min_row_jobs(knobs):
    x, eps, u = _full_inputs(5000)
    cfg = _sigma_cfg("cfg4_B5000", FULL, knobs, "reference", (perturbed_params(make_spec(FULL)), x.bool(), eps, u))
    _check_at(cfg, 5000, "cfg4_B5000", f"sigma={knobs}")


# ------------------------------------------------------------------ Adam hyperparameters and the global step
ADAM = dict(learning_rate=3e-3, beta1=0.5, beta2=0.99, epsilon=1e-4)


def test_adam_hyperparameters_and_set_step():
    """3 steps with non-default Adam hyperparameters against O.adam_tf_step; then set_global_step(1000) and one more step, which
    must use lr_t = lr sqrt(1 - beta2^1001) / (1 - beta1^1001): gmvae_set_step resets the beta-power accumulators."""
    cfg = CONFIGS["tiny_gmvae"]
    spec = make_spec(cfg)
    params = perturbed_params(spec)
    eng = make_engine(cfg, "fp32", **ADAM)
    eng.set_parameters(params)
    st = O.adam_init(params)

    def step(i):
        x, _, eps, u = O.synthetic_batch(spec, cfg["batch"], seed_data=100 + i, seed_noise=200 + i)
        terms, grads = O.loss_and_grads(spec, params, x, eps, u)
        O.adam_tf_step(params, grads, st, lr=ADAM["learning_rate"], beta1=ADAM["beta1"], beta2=ADAM["beta2"], epsilon=ADAM["epsilon"])
        loss = eng.train_step(x, eps=eps, gumbel_u=u)
        assert rel(loss[0].item(), terms["loss"].item()) < 1e-5, i

    def compare(what):
        for got, want, tol in ((eng.parameters(), params, 2e-5), (eng._views(eng.adam_m), st.m, 1e-4), (eng._views(eng.adam_v), st.v, 1e-4)):
            for n, v in got.items():
                r = want[n]
                e = ((v.cpu().double().reshape(r.shape) - r).norm() / r.norm().clamp_min(1e-30)).item()
                assert e < tol, (what, n, e)

    for i in range(3):
        step(i)
    compare("3 steps")
    eng.set_global_step(1000)
    st.t = 1000
    step(3)
    assert eng.global_step == 1001
    compare("step after set_global_step(1000)")
    eng.close()


# ------------------------------------------------------------------ workspace state
# padding everywhere: D = 97, hidden 33 and 7, Z = 3, K = 5 are all rounded up to a multiple of 8 in the row strides
PADDED = dict(model="gmvae", latent_size=3, hidden_sizes=[33, 7], mixture_components=5, batch=64, data_size=97)


def _inference(eng, spec, x, eps, u, n_enc, n_dec):
    """encode / decode / condition (all four networks) on the first rows of the batch."""
    K, Z, D = spec.K, spec.latent_size, spec.data_size
    logits, zm, zs = eng.encode(x[:n_enc], eps=eps[:n_enc], gumbel_u=u[:n_enc])
    y = torch.softmax(torch.randn(n_dec, K, generator=torch.Generator().manual_seed(3)), 1)
    xf = x[:n_dec].float()
    out = {"encode.logits_y": logits, "encode.z_mean": zm, "encode.z_sample": zs, "decode": eng.decode(eps[:n_dec])}
    out["condition.decoder"] = _condition(eng, 0, eps[:n_dec], None, n_dec, D)[0]
    out["condition.encoder.mu"], out["condition.encoder.sigma"] = _condition(eng, 1, xf, y, n_dec, Z, Z)
    out["condition.encoder_y"] = _condition(eng, 2, xf, None, n_dec, K)[0]
    out["condition.prior_gmm.mu"], out["condition.prior_gmm.sigma"] = _condition(eng, 3, y, None, n_dec, Z, Z)
    torch.cuda.synchronize()
    return {k: v.clone() for k, v in out.items()}


def _step(eng, x, eps, u):
    loss = eng.forward_backward(x, eps=eps, gumbel_u=u)
    torch.cuda.synchronize()
    return {"loss": loss.clone(), **{n: g.clone() for n, g in eng.gradients().items()}}


def _assert_equal(a, b, what):
    for k in a:
        assert torch.isfinite(a[k]).all(), (what, k, "reference side not finite")
        assert torch.equal(a[k], b[k]), (what, k, (a[k] - b[k]).abs().max().item())


def _padded_case(precision):
    spec = make_spec(PADDED)
    params = perturbed_params(spec)
    x, _, eps, u = O.synthetic_batch(spec, PADDED["batch"])
    engines = []
    for _ in range(2):
        e = make_engine(PADDED, precision, deterministic=True)
        e.set_parameters(params)
        engines.append(e)
    return spec, params, (x, eps, u), engines


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_nan_filled_workspace(precision):
    """An engine whose workspace holds 0xFF bytes (NaN in fp32 and in bf16) when it is bound computes what a clean one does,
    bit for bit (deterministic mode): no buffer padding that a GEMM contracts over may keep what was in the memory."""
    spec, params, (x, eps, u), (clean, dirty) = _padded_case(precision)
    dirty.workspace.fill_(255)
    ws_ptr = (dirty.workspace.data_ptr() + 255) // 256 * 256
    _lib.check(dirty.lib.gmvae_bind(dirty._h, dirty.params.data_ptr(), dirty.grads.data_ptr(), dirty.adam_m.data_ptr(),
                                    dirty.adam_v.data_ptr(), ws_ptr, dirty.lib.gmvae_workspace_bytes(dirty._h)), "gmvae_bind")
    dirty.set_parameters(params)
    _assert_equal(_step(clean, x, eps, u), _step(dirty, x, eps, u), "training step")
    _assert_equal(_inference(clean, spec, x, eps, u, 50, 40), _inference(dirty, spec, x, eps, u, 50, 40), "inference")
    clean.close(); dirty.close()


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_step_after_inference_calls(precision):
    """encode, decode and condition share z_act, x_act and the hidden buffers with the training step; a step that follows such
    calls (with other row counts) equals the same step on a fresh handle, bit for bit."""
    spec, params, (x, eps, u), (fresh, used) = _padded_case(precision)
    _inference(used, spec, x, eps, u, 17, 40)
    _inference(used, spec, x, eps, u, 64, 9)
    _assert_equal(_step(fresh, x, eps, u), _step(used, x, eps, u), "training step")
    fresh.close(); used.close()
