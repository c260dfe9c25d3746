"""Inference on a GMVAE handle created with objective=marginal (objective M, the K-way marginalised ELBO): gmvae_encode and the
four gmvae_condition's against the oracle's blocks and against an objective-R handle that holds the same parameters; row counts
past what the per-component buffers of an objective-M handle hold (processed in slices); the model accessors, transform and
reconstruct_images on an objective-M model; run_gmvae --objective=marginal end to end, train then eval.

Bars as in tests/test_base_gpu.py: max |got - oracle| / max |oracle| per output below 1e-5 in fp32 and 2e-2 in bf16.  An
objective-M handle runs the same kernels as an objective-R handle on the same inputs, so the two agree to 1e-6 in fp32 and
within the bf16 bar in bf16."""
import json
import os

import numpy as np
import pytest
import torch

from gmvae_b200 import data, runners, utils
from gmvae_b200.base import COND_DECODER, COND_ENCODER, COND_ENCODER_Y, COND_PRIOR_GMM
from oracle import gmvae_oracle as O
from tests.helpers import CONFIGS, make_engine, make_spec, perturbed_params
from tests.test_config_edges_gpu import _condition
from tests.test_runners_gpu import _flags
from tests.test_step_gpu import _record

pytestmark = pytest.mark.gpu

# Measured on one B200 at 1000 W, worst output over the five cases and the slice test: fp32 1.44e-6, bf16 5.68e-3 (the encode
# outputs, where y is sampled from bf16 logits and then rounded to bf16 as encoder_gmm's operand).
TOL = {"fp32": 1e-5, "bf16": 2e-2}
# objective M against objective R, same parameters and inputs: measured 0.0 (bitwise equal) in both precisions, every case
AGREE = {"fp32": 1e-6, "bf16": 2e-2}
# tiny_gmvae, cfg3: the y head fused into the GEMM epilogue (K <= 16); k20_ragged, cfg5_small, m_k128_z8: the unfused y head
CASES = ["tiny_gmvae", "cfg3", "k20_ragged", "m_k128_z8", "cfg5_small"]


def _err(got, ref):
    ref = torch.as_tensor(ref).to(torch.float64)
    return ((got.detach().cpu().double() - ref).abs().max() / ref.abs().max().clamp_min(1e-30)).item()


def _inputs(cfg, n):
    """Parameters and n rows of x, eps [n,Z], u [n,K], a dense y [n,K] and z [n,Z]."""
    spec = make_spec(cfg)
    params = perturbed_params(spec)
    x, _, eps, u = O.synthetic_batch(spec, n)
    g = torch.Generator().manual_seed(3)
    y = torch.softmax(torch.randn(n, spec.K, generator=g, dtype=torch.float64), 1).float()
    z = torch.randn(n, spec.latent_size, generator=g)
    return spec, params, x, eps, u, y, z


def _oracle(spec, params, x, eps, u, y, z):
    L = len(spec.hidden_sizes) + 1
    xd = x.double()
    ly = O.mlp(params, "encoder_y", xd, L)                                                     # gmvae.py:238
    ys = O.gumbel_softmax_sample(ly, u.double(), spec.temperature)                             # :240
    zm, zs = O.normal_params(spec, O.mlp(params, "encoder_gmm", torch.cat([xd, ys], 1), L))    # :246
    logits_x = O.mlp(params, "decoder", z.double(), L) + spec.gen_bias_init
    return {"encode": (ly, zm, zm + zs * eps.double()),
            "decode": (torch.sigmoid(logits_x),),
            COND_DECODER: (logits_x,),
            COND_ENCODER: O.normal_params(spec, O.mlp(params, "encoder_gmm", torch.cat([xd, y.double()], 1), L)),
            COND_ENCODER_Y: (ly,),
            COND_PRIOR_GMM: O.normal_params(spec, O.mlp(params, "prior_gmm", y.double(), 1))}


def _outputs(eng, x, eps, u, y, z):
    """What the engine gives for the keys of _oracle, on the host."""
    n, D, Z, K = x.shape[0], eng.data_size, eng.latent_size, eng.mixture_components
    out = {"encode": eng.encode(x, eps=eps, gumbel_u=u), "decode": (eng.decode(z),),
           COND_DECODER: _condition(eng, COND_DECODER, z, None, n, D)[:1],
           COND_ENCODER: _condition(eng, COND_ENCODER, x.float(), y, n, Z, Z),
           COND_ENCODER_Y: _condition(eng, COND_ENCODER_Y, x.float(), None, n, K)[:1],
           COND_PRIOR_GMM: _condition(eng, COND_PRIOR_GMM, y, None, n, Z, Z)}
    torch.cuda.synchronize()
    return {k: tuple(t.cpu() for t in v) for k, v in out.items()}


def _name(key):
    return key if isinstance(key, str) else {COND_DECODER: "decoder", COND_ENCODER: "encoder_gmm", COND_ENCODER_Y: "encoder_y",
                                             COND_PRIOR_GMM: "prior_gmm"}[key]


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("name", CASES)
def test_parity_and_agreement_with_reference_handle(name, precision):
    cfg = CONFIGS[name]
    spec, params, x, eps, u, y, z = _inputs(cfg, cfg["batch"])
    ref = _oracle(spec, params, x, eps, u, y, z)
    got = {}
    for objective in ("marginal", "reference"):
        eng = make_engine(cfg, precision, objective=objective)
        eng.set_parameters(params)
        got[objective] = _outputs(eng, x, eps, u, y, z)
        eng.close()
    vs_oracle, vs_r = {}, {}
    for key, refs in ref.items():
        for i, r in enumerate(refs):
            tag = f"{_name(key)}[{i}]"
            vs_oracle[tag] = _err(got["marginal"][key][i], r)
            vs_r[tag] = _err(got["marginal"][key][i], got["reference"][key][i].double())
    _record(name, {"test": "marginal_infer", "precision": precision, "vs_oracle": vs_oracle, "m_vs_r": vs_r})
    bad = {k: v for k, v in vs_oracle.items() if not v < TOL[precision]}
    assert not bad, (name, precision, "objective-M handle vs oracle", bad)
    bad = {k: v for k, v in vs_r.items() if not v < AGREE[precision]}
    assert not bad, (name, precision, "objective-M handle vs objective-R handle", bad)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_row_slices(precision, monkeypatch):
    """cfg3 (K = 10) with chunks of 51 samples: the per-component buffers hold 510 rows, max_batch is 1024.  Every entry point
    at 1, 510, 511, 1000 and 1024 rows, the last through Engine.decode / encode of max_batch rows."""
    monkeypatch.setenv("GMVAE_M_CHUNK_ROWS", "512")
    cfg = CONFIGS["cfg3"]
    spec, params, x, eps, u, y, z = _inputs(cfg, 1024)
    ref = _oracle(spec, params, x, eps, u, y, z)
    eng = make_engine(cfg, precision, max_batch=1024, objective="marginal")
    eng.set_parameters(params)
    worst = {}
    for n in (1, 510, 511, 1000, 1024):
        got = _outputs(eng, x[:n], eps[:n], u[:n], y[:n], z[:n])
        for key, refs in ref.items():
            for i, r in enumerate(refs):
                e = _err(got[key][i], r[:n])
                worst[f"{_name(key)}[{i}]"] = max(e, worst.get(f"{_name(key)}[{i}]", 0.0))
                assert e < TOL[precision], (precision, n, _name(key), i, e)
    eng.close()
    _record("cfg3_slices_510", {"test": "marginal_infer_slices", "precision": precision, "vs_oracle_worst": worst})


def test_accessors_on_marginal_model():
    """The accessors, transform, reconstruct_images and encoder_y_logits of a model configured with objective=marginal.  The
    reference's run_model body written with the accessors (as test_base_gpu.test_run_model_composed_from_accessors) gives the
    oracle's objective-R terms; the model's own run_model gives the objective-M terms."""
    import gmvae_b200
    cfg = CONFIGS["cfg3"]
    spec = make_spec(cfg)
    m = gmvae_b200.create_gmvae(spec.data_size, spec.latent_size, mixture_components=spec.mixture_components,
                                fcnet_hidden_sizes=list(spec.hidden_sizes), sigma_min=0.0, raw_sigma_bias=0.5, random_seed=11)
    m.configure(precision="fp32", objective="marginal", max_batch=cfg["batch"])
    params = perturbed_params(spec)
    m.engine().set_parameters(params)
    assert m.engine().objective == "marginal"
    x, _, eps, u = O.synthetic_batch(spec, cfg["batch"])
    q_y = m.encoder_y(x)                                              # gmvae.py:238
    y = q_y.sample(u)                                                 # :240
    p_z_given_y = m.prior_gmm(y)                                      # :243
    q_z = m.encoder_gmm(x, y)                                         # :246
    z = q_z.sample(eps)                                               # :248
    p_x_given_z = m.decoder(z)                                        # :251
    nll = -p_x_given_z.log_prob(x).mean()                             # :254
    kl_div_z = (q_z.log_prob(z) - p_z_given_y.log_prob(z)).mean()     # :258
    logits = q_y.distribution.logits                                  # :263
    nent = (torch.softmax(logits, 1) * torch.log_softmax(logits, 1)).sum(1).mean()
    loss = nll + kl_div_z + nent                                      # :267
    ref = O.loss_terms(spec, params, x, eps, u)
    for got, k in ((loss, "loss"), (nll, "nll"), (kl_div_z, "kl_div_z"), (nent, "nent")):
        assert abs(got.item() - ref[k].item()) / abs(ref[k].item()) < 1e-5, k
    assert _err(m.encoder_y_logits(x), ref["logits_y"]) < 1e-5

    z1, z2 = m.transform(x), m.transform(x)                           # device noise: fresh on every call
    assert tuple(z1.shape) == (x.shape[0], spec.latent_size) and torch.isfinite(z1).all()
    assert not torch.equal(z1, z2)
    r = m.reconstruct_images(x)
    assert tuple(r.shape) == tuple(x.shape) and torch.isfinite(r).all() and bool(((r >= 0) & (r <= 1)).all())

    _, _, eps_m, _ = O.synthetic_batch(spec, cfg["batch"], objective="marginal")
    ref_m = O.loss_terms(spec, params, x, eps_m, None, "marginal")
    fused = m.run_model(x, x, None, eps=eps_m)                        # what run_eval reads under --objective=marginal
    assert abs(fused.item() - ref_m["loss"].item()) / abs(ref_m["loss"].item()) < 1e-5
    m.engine().close()


def test_cli_marginal_train_then_eval(tmp_path, monkeypatch):
    """run_gmvae --objective=marginal: training with summaries (cluster_acc, image tiles) and a checkpoint, evaluation under the
    same objective, then the same checkpoint evaluated under objective R (one variable layout)."""
    monkeypatch.setattr(data, "SPLIT_SIZES", {"train": 2048, "test": 300})
    monkeypatch.delenv("GMVAE_MNIST_DIR", raising=False)
    cfg = _flags(tmp_path, "--mode=train", "--model=gmvae", "--objective=marginal", "--max_steps=59")
    eng = runners.run_train(cfg)
    assert eng.objective == "marginal" and eng.global_step == 60
    logdir = runners.logdir_for(cfg)
    recs = [json.loads(l) for l in open(os.path.join(logdir, "summaries.jsonl"))]
    assert [r["step"] for r in recs] == [20, 40, 60]
    assert all("cluster_acc" in r for r in recs)
    assert all(np.isfinite(list(r.values())).all() for r in recs)
    assert recs[-1]["elbo"] > recs[0]["elbo"]
    for name in ("inputs", "reconstructions", "samples"):
        assert os.path.exists(os.path.join(logdir, "image_summaries", name, "step_60.png"))
    assert utils.get_checkpoint_state(logdir)["model_checkpoint_path"] == "model.ckpt-60"
    eng.close()

    res = runners.run_eval(_flags(tmp_path, "--mode=eval", "--model=gmvae", "--objective=marginal", "--split=test"), max_wait=0.0)
    assert res["step"] == 60 and res["z"].shape == (300, 8)
    assert np.isfinite(res["z"]).all() and np.isfinite(res["loss_per_example"])
    for f in ("step_60.png", "step_60_samples.png", "step_60_sample_images.png", "step_60_sample_k_images.png"):
        assert os.path.exists(os.path.join(res["summary_dir"], f)), f

    res_r = runners.run_eval(_flags(tmp_path, "--mode=eval", "--model=gmvae", "--objective=reference", "--split=test"), max_wait=0.0)
    assert res_r["step"] == 60 and np.isfinite(res_r["loss_per_example"])
