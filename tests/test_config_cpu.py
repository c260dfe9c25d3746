"""Create-time validation of the model and optimiser hyperparameters (gmvae_create, before the device probe): a value that
would only show up as NaN or inf in the first step, or a shape objective M cannot run, is refused when the handle is made."""
import math

import pytest

from tests.test_deterministic_cpu import _cfg as _sized_cfg, _create_error


def _cfg(**kw):
    """A valid GMVAE configuration with the hyperparameters of runners.create_model and tf.train.AdamOptimizer, then `kw`."""
    base = dict(sigma_min=0.0, raw_sigma_bias=0.5, gen_bias_init=0.0, temperature=1.0, learning_rate=1e-3, beta1=0.9,
                beta2=0.999, epsilon=1e-8)
    return _sized_cfg(**{**base, **kw})

NAN, INF = math.nan, math.inf

REJECTED = [
    ("temperature", 0.0, "temperature must be finite and > 0"),
    ("temperature", -1.0, "temperature must be finite and > 0"),
    ("temperature", NAN, "temperature must be finite and > 0"),
    ("temperature", INF, "temperature must be finite and > 0"),
    ("sigma_min", -1e-3, "sigma_min must be finite and >= 0"),
    ("sigma_min", NAN, "sigma_min must be finite and >= 0"),
    ("sigma_min", INF, "sigma_min must be finite and >= 0"),
    ("raw_sigma_bias", NAN, "raw_sigma_bias must be finite"),
    ("raw_sigma_bias", -INF, "raw_sigma_bias must be finite"),
    ("gen_bias_init", NAN, "gen_bias_init must be finite"),
    ("gen_bias_init", INF, "gen_bias_init must be finite"),
    ("learning_rate", 0.0, "learning_rate must be finite and > 0"),
    ("learning_rate", -1e-3, "learning_rate must be finite and > 0"),
    ("learning_rate", NAN, "learning_rate must be finite and > 0"),
    ("learning_rate", INF, "learning_rate must be finite and > 0"),
    ("beta1", 1.0, "beta1 must be in [0, 1)"),
    ("beta1", -0.1, "beta1 must be in [0, 1)"),
    ("beta1", NAN, "beta1 must be in [0, 1)"),
    ("beta2", 1.0, "beta2 must be in [0, 1)"),
    ("beta2", -0.1, "beta2 must be in [0, 1)"),
    ("beta2", NAN, "beta2 must be in [0, 1)"),
    ("epsilon", -1e-8, "epsilon must be finite and >= 0"),
    ("epsilon", NAN, "epsilon must be finite and >= 0"),
    ("epsilon", INF, "epsilon must be finite and >= 0"),
]


@pytest.mark.parametrize("field,value,msg", REJECTED, ids=[f"{f}={v}" for f, v, _ in REJECTED])
def test_create_rejects_hyperparameter(field, value, msg):
    assert _create_error(_cfg(**{field: value})) == msg


# values at the edge of each accepted range pass the checks (on a machine without a GPU the device probe fails next)
ACCEPTED = [("temperature", 1e-3), ("sigma_min", 0.0), ("raw_sigma_bias", -3.0), ("gen_bias_init", -1.5), ("learning_rate", 1e-8),
            ("beta1", 0.0), ("beta2", 0.0), ("epsilon", 0.0), ("beta1", 0.999999), ("temperature", 100.0)]


@pytest.mark.parametrize("field,value", ACCEPTED, ids=[f"{f}={v}" for f, v in ACCEPTED])
def test_create_accepts_hyperparameter(field, value):
    err = _create_error(_cfg(**{field: value}))
    assert err is None or "must" not in err, err


def _marginal(hidden, K, Z):
    cfg = _cfg(objective=1, mixture_components=K, latent_size=Z, num_hidden=len(hidden))
    for i, h in enumerate(hidden):
        cfg.hidden_sizes[i] = h
    return cfg


def test_create_rejects_marginal_hidden_not_multiple_of_4():
    # expand_h1_kernel reads encoder_gmm layer 0 in groups of 4; this used to fail on the first step
    assert _create_error(_marginal([34, 20], 10, 8)) == "objective=marginal needs hidden sizes that are multiples of 4"
    assert _create_error(_marginal([33, 7], 10, 8)) == "objective=marginal needs hidden sizes that are multiples of 4"
    err = _create_error(_marginal([36, 7], 10, 8))        # only layer 0 is read that way
    assert err is None or "must" not in err and "marginal" not in err, err


def test_create_rejects_marginal_prior_table_tile():
    # head_z_m_bwd_kernel holds the K x 2Z prior-table gradient and 512 floats in at most 200 KB of shared memory:
    # (512 + 2 K Z) * 4 <= 204800  <=>  K Z <= 25344
    msg = "objective=marginal: mixture_components * latent_size too large for the prior-table gradient tile"
    assert _create_error(_marginal([64], 128, 256)) == msg
    assert _create_error(_marginal([64], 100, 254)) == msg            # K Z = 25400
    err = _create_error(_marginal([64], 99, 256))                      # K Z = 25344: fits exactly
    assert err is None or "marginal" not in err, err
    err = _create_error(_cfg(objective=0, mixture_components=128, latent_size=256))   # objective R has no such tile
    assert err is None or "marginal" not in err, err


def test_zero_initialised_config_is_rejected():
    # a struct left at zero has temperature 0 (1/T = inf in the relaxed sample) and learning rate 0: refused before the device probe
    assert _create_error(_sized_cfg()) == "temperature must be finite and > 0"
    assert _create_error(_sized_cfg(temperature=1.0)) == "learning_rate must be finite and > 0"


def test_deterministic_checks_come_first():
    # the deterministic-mode checks run before the hyperparameter checks: their messages do not depend on the other fields
    assert _create_error(_sized_cfg(deterministic=2)) == "deterministic must be 0 or 1"
    assert _create_error(_cfg(deterministic=2)) == "deterministic must be 0 or 1"
