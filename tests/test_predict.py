"""The float64 prediction oracle (tests/predict_oracle.py) on the CPU: against the literal per-channel oracle, against the
outputs of the reference source (reference_golden.npz), and the product's prediction host logic against it.

The GPU parity tests (tests/test_gpu_predict.py) measure the CUDA path against this oracle, so it is pinned here first.
"""
import os

import numpy as np
import pytest
import torch

import predict_oracle as po
import refs
from ard_oracle import ARDOracleBackend, kernel_value
from conftest import GOLDEN, MNIST_FIXTURE, rel_err
from oracle import svgp_literal as lit
import svgp_vae_b200 as pkg
from svgp_vae_b200 import backend, configs

F64 = torch.float64
SE, M52, LINEAR, COSINE, ARD = 1, 7, 3, 4, 16


def _literal_kernel(o):
    """kern(x, y, diag) of a literal oracle object on rows in its inducing-point layout (see _inducing_layout)."""
    return lambda x, y, diag=False: o.kernel_matrix(x, y, True, True, diag)


def _inducing_layout(kind, o, aux):
    """Data rows rewritten in the inducing-row layout, so that one kernel function serves every pair of row sets."""
    aux = aux.to(F64)
    if kind == "sprites":                         # [action id | character] -> [action vector | character]
        return torch.cat([o.GPLVM_action[aux[:, 0].long()], aux[:, 1:]], 1)
    out = aux.clone()                             # mnist: [id, angle, pca] -> [id, angle, object vector of id]
    out[:, 2:] = o.object_vectors[aux[:, 0].long()]
    return out


class _LiteralProduct(lit.MiniBatchSVGP):
    """The literal mini-batch SVGP with a productSVGP kernel (Matern, ARD) from tests/ard_oracle.py."""

    def __init__(self, Z, spec, hyp, jitter, N_train, L):
        super().__init__(False, False, Z, "o", jitter, N_train, F64, L)
        self.spec, self.hyp = spec, torch.as_tensor(hyp, dtype=F64)

    def kernel_matrix(self, x, y, x_inducing=True, y_inducing=True, diag_only=False):
        return kernel_value(self.spec, x, y, self.hyp, pairwise=not diag_only)


def _literal_precompute(o, kern, Z, X, means, vars_):
    """Per channel, as make_reference_golden.py feeds SVGPVAE_model.py:1004-1019."""
    mts, sis = [], []
    K_mm, K_nm = kern(Z, Z), kern(X, Z)
    for l in range(means.shape[1]):
        prec = lit.recip_no_nan(vars_[:, l].double())
        si = torch.linalg.inv(K_mm + K_nm.T @ (K_nm * prec[:, None]))
        mts.append(si @ (K_nm.T @ (prec * means[:, l].double())))
        sis.append(si)
    return torch.stack(mts), torch.stack(sis)


def _ard_case(n=300, M=40, L=3, n_test=70):
    cfg = configs.sweep_inputs(n, M, L)
    spec = (M52 | ARD, 4, SE, 4)
    hyp = torch.tensor([0.9, 1.0, 1.2, 1.1, 0.35, 2.9, 1.3, 0.6, 1.0, 1.0, 1.0, 1.0], dtype=F64)
    g = torch.Generator().manual_seed(5)
    Xt = cfg["aux"].double()[:n_test] + 0.1 * torch.randn(n_test, 8, generator=g, dtype=F64)
    return cfg, spec, hyp, Xt


def test_oracle_matches_literal_per_channel():
    """Batched oracle == literal per-channel oracle (1e-10): sprites72 precompute and precomputed prediction, mnist
    conditional generation, and all three entry points for a Matern|ARD x SE product."""
    # sprites72: precompute + prediction from it
    cfg = configs.sprites_inputs(M=72, L=4)
    o = refs.make_pair("sprites", cfg, "cpu")[0]
    kern, Z, X = _literal_kernel(o), o.inducing_index_points, _inducing_layout("sprites", o, cfg["aux"])
    mt, si = po.precompute(kern, Z, X, cfg["y"], cfg["noise"])
    mt0, si0 = _literal_precompute(o, kern, Z, X, cfg["y"], cfg["noise"])
    assert rel_err(mt, mt0) < 1e-10 and rel_err(si, si0) < 1e-10
    pm, pv = po.predict_from_precomputed(kern, Z, X[:100], mt, si, o.jitter)
    for l in range(4):
        m0, B0 = o.approximate_posterior_params_precomputed_GP_posterior_params(cfg["aux"][:100].double(), mt[l], si[l])
        assert rel_err(pm[:, l], m0) < 1e-10 and rel_err(pv[:, l], B0) < 1e-10
    # mnist: test rows against the training rows
    cfg = configs.mnist_inputs(MNIST_FIXTURE, L=4)
    o = refs.make_pair("mnist", cfg, "cpu")[0]
    aux = cfg["aux"].double()
    test_aux = aux[:48].clone()
    test_aux[:, 1] += 0.3
    kern, Z = _literal_kernel(o), o.inducing_index_points
    pm, pv = po.posterior_predict(kern, Z, _inducing_layout("mnist", o, test_aux), _inducing_layout("mnist", o, aux),
                                  cfg["y"], cfg["noise"], o.jitter, o.N_train)
    for l in range(4):
        m0, B0, _, _ = o.approximate_posterior_params(test_aux, aux, cfg["y"][:, l].double(), cfg["noise"][:, l].double())
        assert rel_err(pm[:, l], m0) < 1e-10 and rel_err(pv[:, l], B0) < 1e-10
    # Matern|ARD x SE
    cfg, spec, hyp, Xt = _ard_case()
    X, Z = cfg["aux"].double(), torch.from_numpy(cfg["ctor"]["initial_inducing_points"]).double()
    o = _LiteralProduct(Z, spec, hyp, 1e-2, 5000, 3)
    kern = po.spec_kernel(spec, hyp, rows=64)                  # several row blocks
    pm, pv = po.posterior_predict(kern, Z, Xt, X, cfg["y"], cfg["noise"], 1e-2, 5000)
    mt, si = po.precompute(kern, Z, X, cfg["y"], cfg["noise"])
    mt0, si0 = _literal_precompute(o, _literal_kernel(o), Z, X, cfg["y"], cfg["noise"])
    assert rel_err(mt, mt0) < 1e-10 and rel_err(si, si0) < 1e-10
    qm, qv = po.predict_from_precomputed(kern, Z, Xt, mt, si, 1e-2)
    for l in range(3):
        m0, B0, _, _ = o.approximate_posterior_params(Xt, X, cfg["y"][:, l].double(), cfg["noise"][:, l].double())
        assert rel_err(pm[:, l], m0) < 1e-10 and rel_err(pv[:, l], B0) < 1e-10
        Kinv = torch.linalg.inv(kern(Z, Z) + 1e-2 * torch.eye(40, dtype=F64))
        K_bm = kern(Xt, Z)
        B1 = kern(Xt, Xt, diag=True) + torch.diagonal(-(K_bm @ Kinv @ K_bm.T) + K_bm @ si0[l] @ K_bm.T)
        assert rel_err(qm[:, l], K_bm @ mt0[l]) < 1e-10 and rel_err(qv[:, l], B1) < 1e-10


def test_oracle_reproduces_reference_source():
    """The oracle reproduces the reference source's own outputs (reference_golden.npz) to 1e-10."""
    gold = np.load(os.path.join(GOLDEN, "reference_golden.npz"))
    T = lambda k: torch.from_numpy(gold[k])
    cfg = configs.sprites_inputs(M=72, L=4)
    o = refs.make_pair("sprites", cfg, "cpu")[0]
    kern, Z, X = _literal_kernel(o), o.inducing_index_points, _inducing_layout("sprites", o, cfg["aux"])
    mt, si = po.precompute(kern, Z, X, cfg["y"], cfg["noise"])
    assert rel_err(mt, T("sprites72/precomp_mean_terms")) < 1e-10 and rel_err(si, T("sprites72/precomp_inv_sigma")) < 1e-10
    pm, pv = po.predict_from_precomputed(kern, Z, X[:100], T("sprites72/precomp_mean_terms"), T("sprites72/precomp_inv_sigma"),
                                         o.jitter)
    assert rel_err(pm, T("sprites72/precomp_p_m")) < 1e-10 and rel_err(pv, T("sprites72/precomp_p_v")) < 1e-10
    cfg = configs.mnist_inputs(MNIST_FIXTURE, L=4)
    o = refs.make_pair("mnist", cfg, "cpu")[0]
    aux = cfg["aux"].double()
    test_aux = aux[:48].clone()
    test_aux[:, 1] += 0.3
    pm, pv = po.posterior_predict(_literal_kernel(o), o.inducing_index_points, _inducing_layout("mnist", o, test_aux),
                                  _inducing_layout("mnist", o, aux), cfg["y"], cfg["noise"], o.jitter, o.N_train)
    assert rel_err(pm, T("mnist/cgen_p_m")) < 1e-10 and rel_err(pv, T("mnist/cgen_p_v")) < 1e-10


@pytest.fixture
def ard_backend():
    old = backend.set_backend_for_tests(ARDOracleBackend())
    yield
    backend.set_backend_for_tests(old)


def test_prediction_host_logic_against_oracle(ard_backend):
    """predict.py on the float64 stand-in backend against the oracle: a Matern|ARD x SE product with zero training
    variances (reciprocal_no_nan gives p = 0) and test points placed far from every inducing point (K_xm = 0 exactly)."""
    cfg, spec, hyp, Xt = _ard_case()
    Xt[:10] += 1e3
    noise = cfg["noise"].clone()
    noise[::37, 1] = 0.0
    s = pkg.productSVGP(**cfg["ctor"], kind_a="matern52", kind_b="se", amplitude=(0.9, 1.2),
                        length_scale=(hyp[4:8].tolist(), 1.1))
    assert s._spec() == spec
    hyp = s._hyp().detach().double()                           # the model's float32 values
    kern, Z, X = po.spec_kernel(spec, hyp), torch.from_numpy(cfg["ctor"]["initial_inducing_points"]).double(), cfg["aux"]
    pm0, pv0 = po.posterior_predict(kern, Z, Xt, X, cfg["y"], noise, s.jitter, s.N_train)
    pm, pv = pkg.posterior_predict(s, Xt.float(), X, cfg["y"], noise)
    assert rel_err(pm, pm0) < 2e-5 and rel_err(pv, pv0) < 2e-5
    K_xx = kernel_value(spec, Xt[:10], Xt[:10], hyp, pairwise=False).float()
    assert (pm[:10] == 0).all() and torch.equal(pv[:10], K_xx[:, None].expand(-1, 3))
    mt0, si0 = po.precompute(kern, Z, X, cfg["y"], noise)
    mt, si = pkg.precompute_GP_params_SVGPVAE(cfg["y"], noise, X, s)
    assert rel_err(mt, mt0) < 2e-5 and rel_err(si, si0) < 2e-5
    qm0, qv0 = po.predict_from_precomputed(kern, Z, Xt, mt0, si0, s.jitter)
    for Kinv in (None, torch.linalg.inv(kern(Z, Z) + s.jitter * torch.eye(40, dtype=F64))):
        qm, qv = pkg.predict_from_precomputed(s, Xt.float(), mt0, si0, K_mm_inv=Kinv)
        assert rel_err(qm, qm0) < 2e-5 and rel_err(qv, qv0) < 2e-5
