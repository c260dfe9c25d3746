"""Create-time bound on mixture_components: up to 1024 for the GMVAE under objective R (the wide q(y|x) heads), 128 for VAE_GMP
and objective M.  The checks run before the device probe, so they hold without a GPU."""
import pytest

from tests.test_deterministic_cpu import _create_error
from tests.test_config_cpu import _cfg


def _accepted(err):
    # on a machine without a GPU the device probe fails next; with one the handle is created
    return err is None or "must" not in err


@pytest.mark.parametrize("K", [129, 500, 1024])
def test_gmvae_reference_accepts_wide_k(K):
    err = _create_error(_cfg(mixture_components=K))
    assert _accepted(err), err
    assert err is None or "no CUDA device" in err, err


@pytest.mark.parametrize("deterministic", [0, 1])
def test_gmvae_reference_rejects_past_1024(deterministic):
    assert _create_error(_cfg(mixture_components=1025, deterministic=deterministic)) == "mixture_components must be in [1,1024]"
    assert _create_error(_cfg(mixture_components=0)) == "mixture_components must be in [1,1024]"


def test_vae_gmp_keeps_128():
    assert _create_error(_cfg(model=1, mixture_components=129)) == "mixture_components must be in [1,128]"
    assert _accepted(_create_error(_cfg(model=1, mixture_components=128)))


def test_marginal_keeps_128():
    assert _create_error(_cfg(objective=1, mixture_components=129)) == "mixture_components must be in [1,128]"
    assert _accepted(_create_error(_cfg(objective=1, mixture_components=128)))


def test_vae_ignores_mixture_components():
    assert _accepted(_create_error(_cfg(model=0, mixture_components=5000)))
