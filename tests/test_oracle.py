"""Pins the CPU oracle: closed-form known answers (SURVEY.md §8c KAT-1..6), an independent
torch.distributions restatement, and finite differences of the oracle's own autograd graph."""
import math

import pytest
import torch
import torch.distributions as td

from oracle import gmvae_oracle as O

F64 = torch.float64


def zero_params(spec):
    return {n: torch.zeros(s, dtype=F64) for n, s in O.param_shapes(spec)}


def test_kat1_gmvae_zero_weights():
    for K, loss_ref in ((10, 541.1248044660031), (50, 539.5153665535689)):
        spec = O.Spec("gmvae", latent_size=64, hidden_sizes=[32, 32], mixture_components=K)
        x, _, eps, u = O.synthetic_batch(spec, 7)
        t = O.loss_terms(spec, zero_params(spec), x, eps, u)
        assert abs(t["nll"].item() - 784 * math.log(2)) < 1e-10
        assert abs(t["nll"].item() - 543.4273895589971) < 1e-10
        assert abs(t["kl_div_z"].item()) < 1e-12
        assert abs(t["nent"].item() + math.log(K)) < 1e-12
        assert abs(t["loss"].item() - loss_ref) < 1e-10
        tm = O.loss_terms(spec, zero_params(spec), x, torch.randn(7, K, 64), u, objective="marginal")
        assert abs(tm["loss"].item() - loss_ref) < 1e-10 and abs(tm["kl_div_z"].item()) < 1e-12


def test_kat2_vae_zero_weights():
    spec = O.Spec("vae", latent_size=64, hidden_sizes=[16])
    x, _, eps, _ = O.synthetic_batch(spec, 5)
    t = O.loss_terms(spec, zero_params(spec), x, torch.zeros_like(eps))
    sigma = math.log1p(math.exp(0.5))
    assert abs(sigma - 0.9740769841801067) < 1e-15
    assert abs(t["kl_div_z"].item() - 1.680956112879789) < 1e-12
    assert abs(t["loss"].item() - 545.1083456718769) < 1e-10


def test_kat3_vae_gmp_zero_weights():
    spec = O.Spec("vae_gmp", latent_size=64, hidden_sizes=[16], mixture_components=10)
    x, _, eps, _ = O.synthetic_batch(spec, 5)
    t = O.loss_terms(spec, zero_params(spec), x, torch.zeros_like(eps))
    assert abs(t["kl_div_z"].item() + 21.77587080434673) < 1e-11
    assert abs(t["loss"].item() - 521.6515187546504) < 1e-10


def test_kat4_logq_identity():
    g = torch.Generator().manual_seed(0)
    mu = torch.randn(9, 64, generator=g, dtype=F64)
    sg = torch.rand(9, 64, generator=g, dtype=F64) + 0.1
    eps = torch.randn(9, 64, generator=g, dtype=F64)
    z = mu + sg * eps
    a = O.mvn_diag_log_prob(z, mu, sg)
    b = -0.5 * (eps ** 2).sum(-1) - sg.log().sum(-1) - 32 * O.LOG_2PI
    assert (a - b).abs().max().item() < 1e-12


def test_kat5_xavier_limits():
    want = {(784, 512): 0.068041, (794, 512): 0.067780, (512, 512): 0.076547, (512, 128): 0.096825,
            (512, 10): 0.107211, (10, 128): 0.208514, (64, 512): 0.102062, (10, 64): 0.284747,
            (10,): 0.547723}
    for shape, lim in want.items():
        assert abs(O.glorot_limit(shape) - lim) < 1e-6
    spec = O.Spec("gmvae")
    p = O.init_params(spec)
    for n, s in O.param_shapes(spec):
        if n.endswith("/b"):
            assert p[n].abs().max() == 0
        else:
            assert p[n].abs().max() <= O.glorot_limit(s)
            assert p[n].abs().max() > 0.95 * O.glorot_limit(s)


def test_kat6_adam_tf_form():
    p = {"w": torch.zeros(3, dtype=F64)}
    g = {"w": torch.tensor([1.0, -2.0, 1e-6], dtype=F64)}
    st = O.adam_init(p)
    O.adam_tf_step(p, g, st)
    lr1 = 1e-3 * math.sqrt(1 - 0.999) / (1 - 0.9)
    assert abs(lr1 - 3.1622776601683816e-4) < 1e-18
    assert abs(p["w"][0].item() + 9.99999683772334e-4) < 1e-15
    for i, gi in enumerate([1.0, -2.0, 1e-6]):
        want = -lr1 * 0.1 * gi / (math.sqrt(0.001 * gi * gi) + 1e-8)
        assert abs(p["w"][i].item() - want) < 1e-15
    assert st.t == 1


def test_param_counts():
    # SURVEY.md §8(a8)
    def count(spec):
        return sum(math.prod(s) for _, s in O.param_shapes(spec))
    assert count(O.Spec("vae")) == 1428368
    assert count(O.Spec("vae_gmp")) == 1429658
    assert count(O.Spec("gmvae")) == 2104602
    assert count(O.Spec("gmvae", latent_size=128, hidden_sizes=[1024, 1024], mixture_components=50)) == 6070082


def _td_reference(spec, params, x, eps, u):
    """Independent restatement through torch.distributions (never shares code with loss_terms)."""
    x = x.to(F64)
    L = len(spec.hidden_sizes) + 1
    sp = torch.nn.functional.softplus

    def net(name, h):
        return O.mlp(params, name, h, L if name != "prior_gmm" else 1)

    def normal(outs):
        mu, raw = outs.chunk(2, 1)
        return td.Independent(td.Normal(mu, torch.clamp_min(sp(raw + spec.raw_sigma_bias, threshold=1e9), spec.sigma_min)), 1)

    if spec.model == "gmvae":
        ly = net("encoder_y", x)
        g = td.Gumbel(torch.zeros((), dtype=F64), torch.ones((), dtype=F64)).icdf(u.to(F64))
        y = torch.softmax((ly + g) / spec.temperature, -1)
        pz = normal(net("prior_gmm", y))
        qz = normal(net("encoder_gmm", torch.cat([x, y], 1)))
        z = qz.base_dist.loc + qz.base_dist.scale * eps.to(F64)
        px = td.Independent(td.Bernoulli(logits=net("decoder", z)), 1)
        nll = -px.log_prob(x).mean()
        kl = (qz.log_prob(z) - pz.log_prob(z)).mean()
        nent = -td.Categorical(logits=ly).entropy().mean()
        return nll + kl + nent, nll, kl, nent
    qz = normal(net("encoder", x))
    z = qz.base_dist.loc + qz.base_dist.scale * eps.to(F64)
    px = td.Independent(td.Bernoulli(logits=net("decoder", z)), 1)
    nll = -px.log_prob(x).mean()
    if spec.model == "vae":
        pz = td.Independent(td.Normal(torch.zeros(spec.latent_size, dtype=F64), 1.0), 1)
    else:
        pz = td.MixtureSameFamily(td.Categorical(logits=params["mixture_logits"]),
                                  td.Independent(td.Normal(params["loc"], sp(params["raw_scale_diag"], threshold=1e9)), 1))
    kl = (qz.log_prob(z) - pz.log_prob(z)).mean()
    return nll + kl, nll, kl, torch.zeros((), dtype=F64)


@pytest.mark.parametrize("model", ["vae", "vae_gmp", "gmvae"])
def test_against_torch_distributions(model):
    spec = O.Spec(model, latent_size=16, hidden_sizes=[48, 40], mixture_components=7)
    params = O.init_params(spec, seed=3)
    for n in params:  # non-zero biases so every path is exercised
        if n.endswith("/b"):
            params[n] = 0.1 * torch.randn(params[n].shape, dtype=F64, generator=torch.Generator().manual_seed(len(n)))
    x, _, eps, u = O.synthetic_batch(spec, 11)
    t = O.loss_terms(spec, params, x, eps, u)
    loss, nll, kl, nent = _td_reference(spec, params, x, eps, u)
    for a, b in ((t["loss"], loss), (t["nll"], nll), (t["kl_div_z"], kl), (t["nent"], nent)):
        assert abs(a.item() - b.item()) <= 1e-10 * max(1.0, abs(b.item()))


# a non-default set of every model hyperparameter; sigma_min clamps part of the scales, none of them within 1e-3 of the kink
KNOBS_FD = dict(temperature=0.7, sigma_min=0.55, raw_sigma_bias=-0.2, gen_bias_init=-0.8)
FD_CASES = [pytest.param(m, o, {}, id=f"{m}-{o}") for m, o in (("vae", "reference"), ("vae_gmp", "reference"), ("gmvae", "reference"),
                                                              ("gmvae", "marginal"))]
FD_CASES += [pytest.param(m, o, KNOBS_FD, id=f"{m}-{o}-knobs") for m, o in (("vae_gmp", "reference"), ("gmvae", "reference"),
                                                                             ("gmvae", "marginal"))]


@pytest.mark.parametrize("model,objective,knobs", FD_CASES)
def test_finite_differences(model, objective, knobs):
    spec = O.Spec(model, data_size=20, latent_size=4, hidden_sizes=[6, 5], mixture_components=3, **knobs)
    params = O.init_params(spec, seed=5)
    for n in params:
        if n.endswith("/b"):
            params[n] = 0.2 * torch.randn(params[n].shape, dtype=F64, generator=torch.Generator().manual_seed(len(n)))
    x, _, eps, u = O.synthetic_batch(spec, 6, objective=objective)
    if knobs:
        # the clamp is active and every scale is away from its kink, where the loss is not differentiable
        t = O.loss_terms(O.Spec(model, data_size=20, latent_size=4, hidden_sizes=[6, 5], mixture_components=3,
                                **dict(knobs, sigma_min=0.0)), params, x, eps, u, objective)
        s = torch.cat([t[k].reshape(-1) for k in ("sigma_q", "sigma_p") if k in t])
        assert 0.1 < (s < spec.sigma_min).double().mean().item() < 0.9
        assert (s - spec.sigma_min).abs().min().item() > 1e-3
    _, grads = O.loss_and_grads(spec, params, x, eps, u, objective)
    g = torch.Generator().manual_seed(9)
    h = 1e-6
    for n, p in params.items():
        for _ in range(3):
            idx = tuple(int(torch.randint(0, s, (1,), generator=g)) for s in p.shape)
            pp = {k: v.clone() for k, v in params.items()}
            pm = {k: v.clone() for k, v in params.items()}
            pp[n][idx] += h
            pm[n][idx] -= h
            fd = (O.loss_terms(spec, pp, x, eps, u, objective)["loss"] - O.loss_terms(spec, pm, x, eps, u, objective)["loss"]) / (2 * h)
            assert abs(fd.item() - grads[n][idx].item()) < 1e-6 * max(1.0, abs(fd.item())), (n, idx)


def test_marginal_matches_reference_at_one_hot():
    """SURVEY.md A.4: objective M's component-k reconstruction equals objective R forced to y=e_k."""
    spec = O.Spec("gmvae", data_size=30, latent_size=5, hidden_sizes=[8], mixture_components=4)
    params = O.init_params(spec, seed=1)
    x, _, eps, u = O.synthetic_batch(spec, 3, objective="marginal")
    K = 4
    tm = O.loss_terms(spec, params, x, eps, u, "marginal")
    rec = O.bernoulli_log_prob(x.to(F64)[:, None, :].expand(3, K, 30).reshape(3 * K, 30), tm["logits_x"]).reshape(3, K)
    for k in range(K):
        uk = torch.full((3, K), 1e-30, dtype=F64)
        uk[:, k] = 1 - 1e-16   # Gumbel noise that forces the relaxed sample to e_k
        tr = O.loss_terms(spec, params, x, eps[:, k], uk)
        assert (tr["y"][:, k] - 1).abs().max() < 1e-12
        rk = O.bernoulli_log_prob(x.to(F64), tr["logits_x"])
        assert (rk - rec[:, k]).abs().max() < 1e-9


def test_global_batch_sharding_sums():
    """§8(e): shards scaled by 1/B_global sum to the single-batch loss and gradients."""
    spec = O.Spec("gmvae", data_size=40, latent_size=6, hidden_sizes=[12, 12], mixture_components=5)
    params = O.init_params(spec, seed=2)
    x, _, eps, u = O.synthetic_batch(spec, 10)
    t, g = O.loss_and_grads(spec, params, x, eps, u)
    t0, g0 = O.loss_and_grads(spec, params, x[:4], eps[:4], u[:4], global_batch=10)
    t1, g1 = O.loss_and_grads(spec, params, x[4:], eps[4:], u[4:], global_batch=10)
    assert abs((t0["loss"] + t1["loss"] - t["loss"]).item()) < 1e-10
    for n in g:
        assert (g0[n] + g1[n] - g[n]).abs().max().item() < 1e-12


def test_bf16_rounding_model_explains_gradient_gap():
    """A 2^-9 relative rounding of stored activations changes the LOSS by < 1e-4 but individual
    gradient tensors by > 1e-3 (ReLU-mask flips): the reason tests/test_step_gpu.py compares bf16
    gradients under the rounding model and only bounds the distance to the exact oracle."""
    from tests.helpers import CONFIGS, Bf16Model, make_spec, perturbed_params
    cfg = CONFIGS["tiny_gmvae"]
    spec = make_spec(cfg)
    params = perturbed_params(spec)
    x, _, eps, u = O.synthetic_batch(spec, cfg["batch"])
    t0, g0 = O.loss_and_grads(spec, params, x, eps, u)
    t1, g1 = O.loss_and_grads(spec, params, x, eps, u, q=Bf16Model(True))
    assert abs(t0["loss"].item() - t1["loss"].item()) / t0["loss"].item() < 2e-3
    worst = max(((g1[n] - g0[n]).norm() / g0[n].norm()).item() for n in g0)
    assert 1e-3 < worst < 0.1


# --------------------------------------------------------------------------- hyperparameter sensitivity
def _knob_cases():
    """The hyperparameter cases of tests/test_config_edges_gpu.py on their small shapes: (id, cfg, objective, knob values)."""
    from tests.helpers import CONFIGS
    out = []
    for name in ("cfg3", "k20_ragged"):
        for T in (0.5, 2.0):
            out.append((f"{name}-T={T}", CONFIGS[name], "reference", dict(temperature=T)))
    for name, obj in (("cfg1", "reference"), ("tiny_gmp", "reference"), ("cfg3", "reference"), ("tiny_gmvae", "marginal")):
        out.append((f"{name}-{obj}-gen_bias_init", CONFIGS[name], obj, dict(gen_bias_init=-1.5)))
        for knobs in ("dropin", "active"):
            out.append((f"{name}-{obj}-sigma={knobs}", CONFIGS[name], obj, knobs))
    return out


KNOB_CASES = _knob_cases()
FP32_BAR = 1e-5          # what the GPU tests hold the fp32 validation mode to, per loss term and per gradient tensor


# the tensors each knob acts on first: the networks whose output it enters
DIRECT = {"temperature": ("encoder_y_fcnet/",), "gen_bias_init": ("decoder_fcnet/",),
          "sigma": ("encoder_fcnet/", "encoder_gmm_fcnet/", "prior_gmm_fcnet/")}


@pytest.mark.parametrize("case", KNOB_CASES, ids=[c[0] for c in KNOB_CASES])
def test_knob_values_move_the_oracle(case):
    """The oracle at each knob value of the GPU tests and at the default differs by at least 20 x the fp32 bar in the loss and in
    every gradient tensor of the networks the knob acts on (a kernel that ignored the knob fails there), and by at least 10 x the
    bar in every other tensor it reaches (one equal to 1e-12 is not reached, e.g. the prior's gradients by gen_bias_init).  Loss
    terms other than the loss are not held: the relaxed sample reaches nll through z only, and T = 0.5 moves it by 2e-6 on cfg3."""
    from tests.helpers import active_clamp, make_spec, perturbed_params
    cid, cfg, obj, knobs = case
    spec0 = make_spec(cfg)
    params = perturbed_params(spec0)
    x, _, eps, u = O.synthetic_batch(spec0, cfg["batch"], objective=obj)
    if knobs == "dropin":
        knobs = dict(sigma_min=0.001, raw_sigma_bias=0.25)
    elif knobs == "active":
        knobs = {k: v for k, v in active_clamp(cfg, params, x, eps, u, obj).items() if k in ("sigma_min", "raw_sigma_bias")}
    direct = DIRECT["sigma" if "sigma_min" in knobs else next(iter(knobs))]
    t0, g0 = O.loss_and_grads(spec0, params, x, eps, u, obj)
    t1, g1 = O.loss_and_grads(make_spec(dict(cfg, **knobs)), params, x, eps, u, obj)
    assert abs(t1["loss"].item() - t0["loss"].item()) / abs(t0["loss"].item()) > 20 * FP32_BAR
    n_direct = 0
    for n in g0:
        d = ((g1[n] - g0[n]).norm() / g0[n].norm().clamp_min(1e-30)).item()
        if n.startswith(direct):
            n_direct += 1
            assert d > 20 * FP32_BAR, (cid, n, d)
        else:
            assert d < 1e-12 or d > 10 * FP32_BAR, (cid, n, d)
    assert n_direct >= 2
