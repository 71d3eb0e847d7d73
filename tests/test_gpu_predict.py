"""The prediction entry points (posterior_predict, precompute_GP_params_SVGPVAE, predict_from_precomputed) on the B200
against the float64 prediction oracle evaluated on the GPU (tests/predict_oracle.py through
tests/probes/parity_predict.py), at the sizes where they run on the tensor cores.

The row sets of posterior_predict land on the tensor-core path from 2048 rows on (backend.tc_min_rows): the shapes put
both the training rows and the test rows there, and one case each puts only the training rows there or has a single test
point.  M = 1000 gives ragged tiles; M = 4096 is where the step's forward SYRK takes thirteen digit-plane pairs.

Every output is held to 1e-4 of max |oracle tensor|.  Test points far from every inducing point (every feature shifted by
1e3) have K_xm = 0 exactly, in float64 and in fp32, so there p_m = 0 and p_v = K_xx exactly.  With the training rows as
test rows, posterior_predict is the training step's computation and equals its p_m / p_v to 1e-6.
"""
import os
import sys

import pytest
import torch

from conftest import rel_err
import svgp_vae_b200 as pkg

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "probes"))
import parity_predict as pp  # noqa: E402

pytestmark = pytest.mark.gpu
TOL = 1e-4

# (n_train, n_test, M, L)
SE_SHAPES = [
    (4096, 2304, 256, 3),
    (65536, 4096, 1024, 4),
    (32768, 2048, 2048, 2),
    (16384, 2048, 4096, 2),
    (30000, 2500, 1000, 3),
    (8192, 2048, 1024, 64),
    (8192, 1, 1024, 2),                 # a single test point
    (8192, 1000, 1024, 2),              # test rows on the SIMT path, training rows on the tensor cores
]


def _check(out, keys):
    bad = {k: out[k] for k in keys if not out[k] < TOL}
    assert not bad, (bad, out)


@pytest.mark.parametrize("shape", SE_SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_posterior_predict_se(cuda_backend, shape):
    """Product SE (the SE44 integer builder), test points near the training data."""
    _check(pp.run(*shape, kind="se", placement="near", precomputed=False), ("p_m", "p_v"))


@pytest.mark.parametrize("kind,shape", [("m52ard_se", (8192, 2304, 1024, 3)), ("m52ard_se", (32768, 2048, 2048, 2)),
                                        ("lin_cos", (8192, 2304, 256, 3)), ("lin_cos", (32768, 2048, 256, 2))],
                         ids=lambda v: v if isinstance(v, str) else "x".join(map(str, v)))
def test_posterior_predict_kernels(cuda_backend, kind, shape):
    """Matern 5/2 with ARD x SE (the generic builder) and linear x cosine (entries of both signs; at M = 256, the largest M
    at which its rank-256 kernel on K1's 32 features leaves the prediction well posed, see parity_predict.KINDS)."""
    _check(pp.run(*shape, kind=kind, placement="near", precomputed=False), ("p_m", "p_v"))


def _far_rows(placement, n):
    return torch.arange(n, device="cuda") if placement == "far" else torch.arange(0, n, 3, device="cuda")


@pytest.mark.parametrize("placement", ["far", "mix"])
@pytest.mark.parametrize("kind", ["se", "m52ard_se"])
@pytest.mark.parametrize("M", [1024, 2048])
def test_far_test_points(cuda_backend, kind, placement, M):
    """Test points with K_xm = 0 (all of them, or every third row inside the tensor-core tiles): p_m = 0 and p_v = K_xx
    exactly, from posterior_predict and from predict_from_precomputed; the other rows at the oracle's tolerance."""
    n_train, n_test, L = 8192, 2304, 2
    s, X, y, nz, Xt = pp.make_case(n_train, n_test, M, L, kind=kind, placement=placement)
    kern, Z = pp.oracle_kernel(s), s.inducing_index_points.detach().double()
    far = _far_rows(placement, n_test)
    assert (kern(Xt[far], Z) == 0).all()
    K_xx = cuda_backend.kernel_diag_fwd(s._spec(), Xt, Xt, s._hyp().detach().float().contiguous())[far][:, None].expand(-1, L)
    pm0, pv0 = pp.po.posterior_predict(kern, Z, Xt, X, y, nz, s.jitter, s.N_train)
    pm, pv = pkg.posterior_predict(s, Xt, X, y, nz)
    assert (pm[far] == 0).all() and torch.equal(pv[far], K_xx)
    assert rel_err(pm, pm0) < TOL and rel_err(pv, pv0) < TOL
    mt0, si0 = pp.po.precompute(kern, Z, X, y, nz)
    qm0, qv0 = pp.po.predict_from_precomputed(kern, Z, Xt, mt0, si0, s.jitter)
    qm, qv = pkg.predict_from_precomputed(s, Xt, mt0, si0)
    assert (qm[far] == 0).all() and torch.equal(qv[far], K_xx)
    assert rel_err(qm, qm0) < TOL and rel_err(qv, qv0) < TOL


@pytest.mark.parametrize("shape", [(8192, 1024, 4), (16384, 2048, 2), (16384, 4096, 2)], ids=lambda s: "x".join(map(str, s)))
def test_precomputed_posterior(cuda_backend, shape):
    """precompute_GP_params_SVGPVAE (mean_terms, inv_Sigma) and predict_from_precomputed on 2304 test rows, fed the
    oracle's float64 precompute (the function on its own) and the device's."""
    n_train, M, L = shape
    out = pp.run(n_train, 2304, M, L, kind="se", placement="near", precomputed=True)
    _check(out, ("mean_terms", "inv_Sigma", "pfp_p_m", "pfp_p_v", "pfp_dev_p_m", "pfp_dev_p_v"))


def test_posterior_predict_on_training_rows_against_oracle(cuda_backend):
    """Test rows = training rows (the step's own rows), against the oracle."""
    _check(pp.run(8192, 8192, 1024, 4, kind="se", placement="train", precomputed=False), ("p_m", "p_v"))


@pytest.mark.parametrize("shape", [(4096, 256, 3), (32768, 2048, 2), (16384, 4096, 2), (8192, 1024, 64), (1_000_000, 1024, 8)],
                         ids=lambda s: "x".join(map(str, s)))
def test_posterior_predict_is_the_step(cuda_backend, shape):
    """posterior_predict(s, X, X, y, noise) == elbo_step(X, y, noise)[p_m, p_v] to 1e-6, zero variances included (at
    N = 1e6, M = 1024, the headline size, where the float64 oracle is too slow)."""
    N, M, L = shape
    s, X, y, nz, _ = pp.make_case(N, N, M, L, placement="train")
    with torch.no_grad():
        res = s.elbo_step(X, y, nz)
    pm, pv = pkg.posterior_predict(s, X, X, y, nz)
    assert rel_err(pm, res["p_m"]) < 1e-6 and rel_err(pv, res["p_v"]) < 1e-6


def test_zero_variances_carry_no_weight(cuda_backend):
    """Training rows with var = 0 get p = 0 (reciprocal_no_nan), as in the step: changing their means changes nothing."""
    s, X, y, nz, Xt = pp.make_case(8192, 2304, 1024, 2, placement="near")
    zero = nz == 0
    assert zero.any()
    pm, pv = pkg.posterior_predict(s, Xt, X, y, nz)
    pm2, pv2 = pkg.posterior_predict(s, Xt, X, torch.where(zero, y + 5.0, y), nz)
    assert torch.isfinite(pm).all() and torch.isfinite(pv).all()
    assert rel_err(pm2, pm) < 1e-7 and rel_err(pv2, pv) < 1e-7      # the float64 SYRK's summation order is not fixed
