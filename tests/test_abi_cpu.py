"""CPU-side checks of the drop-in boundary: the C-ABI library loads and exports every symbol
include/gmvae_abi.h declares, the host mirrors keep the reference's signatures and defaults,
and the product fails loudly without a GPU (no CPU fallback)."""
import ctypes as C
import inspect
import os
import re

import pytest
import torch

import gmvae_b200
from gmvae_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_functions():
    src = open(os.path.join(ROOT, "include", "gmvae_abi.h")).read()
    return sorted(set(re.findall(r"GMVAE_API[^;(]*?\b(gmvae_\w+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    lib = _lib.load()
    names = header_functions()
    assert len(names) >= 25
    for n in names:
        assert hasattr(lib, n), n
    assert sorted(_lib.SYMBOLS) == names      # binding table and header agree
    assert b"sm_100a" in lib.gmvae_build_info()


def test_config_struct_layout_matches_header():
    # 4 + 3 + 1 + 8 + 1 ints, 8 floats, 1 + 7 ints = 33 x 4 bytes
    assert C.sizeof(_lib.Config) == 4 * (4 + 3 + 1 + 8 + 1 + 8 + 1 + 7)
    assert C.sizeof(_lib.ParamDesc) == 64 + 8 + 4 + 4


@pytest.mark.skipif(torch.cuda.is_available(), reason="CPU-only behaviour")
def test_no_cpu_fallback():
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        gmvae_b200.Engine()
    lib = _lib.load()
    cfg = _lib.Config()
    cfg.abi_version = 1; cfg.model = 2; cfg.precision = 1; cfg.data_size = 784; cfg.latent_size = 8
    cfg.mixture_components = 10; cfg.num_hidden = 1; cfg.hidden_sizes[0] = 64; cfg.max_batch = 16
    cfg.raw_sigma_bias = 0.5; cfg.temperature = 1.0; cfg.learning_rate = 1e-3; cfg.beta1 = 0.9; cfg.beta2 = 0.999; cfg.epsilon = 1e-8
    h = C.c_void_p()
    rc = lib.gmvae_create(C.byref(cfg), C.byref(h))
    assert rc != 0 and b"no CPU fallback" in lib.gmvae_last_error()
    m = gmvae_b200.create_gmvae(784, 8, 10)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m.run_model(torch.zeros(4, 784, dtype=torch.bool), torch.zeros(4, 784, dtype=torch.bool), torch.zeros(4))


def test_create_rejects_bad_config():
    lib = _lib.load()
    h = C.c_void_p()
    cfg = _lib.Config()
    cfg.abi_version = 99
    assert lib.gmvae_create(C.byref(cfg), C.byref(h)) != 0
    assert b"ABI version" in lib.gmvae_last_error()
    cfg.abi_version = 1; cfg.model = 7
    assert lib.gmvae_create(C.byref(cfg), C.byref(h)) != 0


def test_factory_signatures_match_reference():
    # gmvae.py:277-287, vae.py:191-200
    sg = inspect.signature(gmvae_b200.create_gmvae)
    assert list(sg.parameters) == ["data_size", "latent_size", "mixture_components", "fcnet_hidden_sizes",
                                   "hidden_activation_fn", "sigma_min", "raw_sigma_bias", "gen_bias_init",
                                   "temperature", "random_seed"]
    assert sg.parameters["sigma_min"].default == 0.001 and sg.parameters["raw_sigma_bias"].default == 0.25
    assert sg.parameters["mixture_components"].default == 1 and sg.parameters["temperature"].default == 1.0
    sv = inspect.signature(gmvae_b200.create_vae)
    assert list(sv.parameters) == ["data_size", "latent_size", "mixture_components", "fcnet_hidden_sizes",
                                   "hidden_activation_fn", "sigma_min", "raw_sigma_bias", "gen_bias_init", "random_seed"]
    m = gmvae_b200.create_gmvae(784, 8, mixture_components=10)
    assert isinstance(m, gmvae_b200.TrainableGMVAE) and m.mix_components == 10 and m.random_seed is None
    assert m._encoder_gmm.hidden_layer_sizes == [8]          # fcnet_hidden_sizes=None -> [latent_size]
    assert m._prior_gmm.hidden_layer_sizes is None           # gmvae.py:321-327
    assert m._prior_gmm.variable_names() == ["prior_gmm_fcnet/linear_0/w", "prior_gmm_fcnet/linear_0/b"]
    assert m._encoder_y.output_sizes == [8, 10] and m._encoder_gmm.output_sizes == [8, 16]
    v = gmvae_b200.create_vae(784, 8, mixture_components=10, fcnet_hidden_sizes=[32, 32])
    assert isinstance(v, gmvae_b200.TrainableVAE) and v._prior == "mixture"
    assert hasattr(v.prior(), "log_prob") and hasattr(v.prior(), "sample")          # vae.py:41-48: prior() returns a distribution
    for acc in ("prior_gmm", "decoder", "encoder_y", "encoder_gmm"):                 # gmvae.py:49-107
        assert callable(getattr(m, acc))
    for acc in ("prior", "decoder", "encoder"):                                      # vae.py:41-78
        assert callable(getattr(v, acc))
    import gmvae_b200.base as base
    for cls in (base.ConditionalNormal, base.ConditionalBernoulli, base.ConditionalCategorical):
        assert callable(getattr(cls, "condition")) and callable(getattr(cls, "__call__"))
    with pytest.raises(RuntimeError):                                                # not part of a model: no variables to run
        base.ConditionalNormal(size=4, name="free").condition([torch.zeros(2, 3)])
    assert list(inspect.signature(v.run_model).parameters)[:2] == ["images", "targets"]
    assert list(inspect.signature(m.run_model).parameters)[:3] == ["images", "targets", "labels"]
    with pytest.raises(NotImplementedError):
        gmvae_b200.create_vae(784, 8, hidden_activation_fn=torch.tanh)
