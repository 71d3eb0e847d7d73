"""Parity of the prediction entry points (svgp_vae_b200/predict.py) against the float64 prediction oracle
(tests/predict_oracle.py) EVALUATED ON THE GPU.

  posterior_predict           test rows against n_train training rows
  precompute_GP_params_SVGPVAE  mean_terms, inv_Sigma (only for the SE and Matern kinds: without jitter, Sigma_l of a
                              low-rank linear x cosine kernel is singular)
  predict_from_precomputed    on the test rows, fed (a) the oracle's float64 mean_terms / inv_Sigma, (b) the device's

Errors are max |device - oracle| / max |oracle| per output tensor.  Inputs: configs.sweep_inputs(n_train, M, L, seed)
with a few exact zeros in the training variances; test rows X[:n_test] + 0.1 N(0, 1) ("near"), shifted by 1e3 in every
feature ("far": K_xm = 0 exactly), every third row far ("mix") or the training rows themselves ("train").

Usage: python tests/probes/parity_predict.py n_train n_test M L [seed] [kind] [placement] -> one JSON line.
kind: se (the sweep's product SE, SE44 integer builder), m52ard_se (Matern 5/2 with ARD x SE, the generic builder),
lin_cos (linear x cosine on 16 + 16 features, not element-wise non-negative).
"""
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import predict_oracle as po  # noqa: E402
import svgp_vae_b200 as pkg  # noqa: E402
from svgp_vae_b200 import configs  # noqa: E402

F64 = torch.float64
KINDS = {
    "se": dict(),
    "m52ard_se": dict(kind_a="matern52", kind_b="se", length_scale=([0.35, 2.9, 1.3, 0.6], 1.0)),
    "lin_cos": dict(kind_a="linear", kind_b="cosine", dim_a=16, dim_b=16),
}
# linear x cosine has rank dim_a * dim_b: on the sweep's 4 + 4 features (rank 16) the prediction at M = 1024 is so badly
# posed that rounding the kernel entries to fp32 INSIDE the float64 oracle moves p_v by 3.6e-4.  K1 takes at most 32
# features, so this kind runs on 16 + 16 (rank 256) at M = 256, where that rounding moves p_v by 4.7e-6
FAR = 1e3


def rel(a, b):
    a, b = a.detach().double(), b.detach().double()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-300))


def make_case(n_train, n_test, M, L, seed=1234, kind="se", placement="near"):
    """-> (model, training rows, means, vars (zeros included), test rows) on the GPU."""
    dev = torch.device("cuda")
    cfg = configs.sweep_inputs(n_train, M, L, device=dev, seed=seed)
    X, y, nz = cfg["aux"], cfg["y"], cfg["noise"].clone()
    kw = dict(KINDS[kind])
    if "dim_a" in kw:                                       # wider features than the sweep's, same seeds
        d = kw["dim_a"] + kw["dim_b"]
        cfg["ctor"].update(dim_a=kw.pop("dim_a"), dim_b=kw.pop("dim_b"),
                           initial_inducing_points=torch.randn(M, d, generator=configs._gen(7)).numpy())
        X = torch.randn(n_train, d, generator=torch.Generator(device=dev).manual_seed(seed), device=dev)
    s = pkg.productSVGP(**cfg["ctor"], **kw).to(dev)
    nz[::97, 0] = 0.0                                       # reciprocal_no_nan: these rows carry no weight
    if placement == "train":
        assert n_test == n_train
        return s, X, y, nz, X
    g = torch.Generator(device=dev).manual_seed(seed + 17)
    Xt = X[:n_test] + 0.1 * torch.randn(n_test, X.shape[1], generator=g, device=dev)
    if placement == "far":
        Xt = Xt + FAR
    elif placement == "mix":
        Xt[::3] += FAR
    else:
        assert placement == "near", placement
    return s, X, y, nz, Xt.contiguous()


def oracle_kernel(s):
    return po.spec_kernel(s._spec(), s._hyp().detach().double())


def run(n_train, n_test, M, L, seed=1234, kind="se", placement="near", precomputed=None):
    s, X, y, nz, Xt = make_case(n_train, n_test, M, L, seed, kind, placement)
    kern, Z = oracle_kernel(s), s.inducing_index_points.detach().double()
    out = dict(n_train=n_train, n_test=n_test, M=M, L=L, kind=kind, placement=placement)
    pm0, pv0 = po.posterior_predict(kern, Z, Xt, X, y, nz, s.jitter, s.N_train)
    pm, pv = pkg.posterior_predict(s, Xt, X, y, nz)
    out["p_m"], out["p_v"] = rel(pm, pm0), rel(pv, pv0)
    del pm0, pv0
    if precomputed if precomputed is not None else kind != "lin_cos":
        mt0, si0 = po.precompute(kern, Z, X, y, nz)
        mt, si = pkg.precompute_GP_params_SVGPVAE(y, nz, X, s)
        out["mean_terms"], out["inv_Sigma"] = rel(mt, mt0), rel(si, si0)
        qm0, qv0 = po.predict_from_precomputed(kern, Z, Xt, mt0, si0, s.jitter)
        qm, qv = pkg.predict_from_precomputed(s, Xt, mt0, si0)
        out["pfp_p_m"], out["pfp_p_v"] = rel(qm, qm0), rel(qv, qv0)
        qm, qv = pkg.predict_from_precomputed(s, Xt, mt, si)
        out["pfp_dev_p_m"], out["pfp_dev_p_v"] = rel(qm, qm0), rel(qv, qv0)
    return out


if __name__ == "__main__":
    a = sys.argv[1:]
    n_train, n_test, M, L = (int(x) for x in a[:4])
    seed = int(a[4]) if len(a) > 4 else 1234
    kind = a[5] if len(a) > 5 else "se"
    placement = a[6] if len(a) > 6 else "near"
    o = run(n_train, n_test, M, L, seed, kind, placement)
    print(json.dumps({k: (float("%.3g" % v) if isinstance(v, float) else v) for k, v in o.items()}), flush=True)
