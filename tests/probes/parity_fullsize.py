"""Parity of the tcgen05 path at (near) full size against the float64 oracle EVALUATED ON THE GPU.

The streamlined oracle (oracle/svgp_streamlined.py) is device-agnostic torch float64; the product-SE kernel matrix is
restated with the |x|^2 + |z|^2 - 2 x.z expansion in float64 (checked here against oracle/tfp_kernels on the first
rows) so that no (N, M, d) tensor is needed.  Usage: python tests/probes/parity_fullsize.py N M L [seed] -> one JSON line."""
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from oracle import svgp_streamlined as st  # noqa: E402
from oracle import tfp_kernels as tfk  # noqa: E402
import svgp_vae_b200 as pkg  # noqa: E402
from svgp_vae_b200 import configs  # noqa: E402

F64 = torch.float64


def se64(a, b, amp, ls):
    d2 = (a * a).sum(1)[:, None] + (b * b).sum(1)[None, :] - 2.0 * (a @ b.T)
    return amp * amp * torch.exp(-0.5 * d2.clamp_min(0.0) / (ls * ls))


def kern64(X, Z, hyp):
    return se64(X[:, :4], Z[:, :4], hyp[0], hyp[1]) * se64(X[:, 4:], Z[:, 4:], hyp[2], hyp[3])


def rel(a, b):
    a, b = a.detach().double(), b.detach().double()
    return float((a - b).abs().max() / b.abs().max())


def upstream(N, L, dev):
    """The seeded cotangents gm, gv (N, L) float64 of J = KL_term + <gm, p_m> + <gv, p_v>."""
    g = torch.Generator(device=dev).manual_seed(0)
    return (torch.randn(N, L, generator=g, device=dev, dtype=F64), torch.randn(N, L, generator=g, device=dev, dtype=F64))


def objective(res, gm, gv, world=1):
    """J of one rank's elbo_step result: its own rows' <gm, p_m> + <gv, p_v> plus the global KL_term / world (the gradient
    convention under a group: the ranks' J sum to the single-process J)."""
    return res["KL_term"] / world + (gm.float() * res["p_m"]).sum().double() + (gv.float() * res["p_v"]).sum().double()


def oracle(cfg, Z0, gm, gv):
    """The streamlined float64 oracle on the GPU at the inputs of configs.sweep_inputs (unit hypers, inducing points Z0):
    -> dict of p_m, p_v, recon_l, kl_l, ce_l, KL_term and the gradients dy, dnoise, dZ, dhyp of J (detached)."""
    dev = gm.device
    N, L = gm.shape
    X = cfg["aux"].double()
    y = cfg["y"].double().requires_grad_(True)
    nz = cfg["noise"].double().requires_grad_(True)
    Z = Z0.detach().double().clone().requires_grad_(True)
    hyp = torch.ones(4, dtype=F64, device=dev, requires_grad=True)
    one = torch.ones((), dtype=F64, device=dev)
    ref_k = tfk.ExponentiatedQuadratic(one, one).matrix(X[:256, :4], Z[:, :4]) * tfk.ExponentiatedQuadratic(one, one).matrix(X[:256, 4:], Z[:, 4:])
    assert rel(kern64(X[:256], Z, hyp), ref_k) < 1e-12
    K_nm, K_mm = kern64(X, Z, hyp), kern64(Z, Z, hyp)
    kappa = (hyp[0] * hyp[2]) ** 2 * torch.ones(N, dtype=F64, device=dev)
    t0 = st.streamlined_terms(K_nm, K_mm, kappa, y, nz, float(N), cfg["ctor"]["jitter"])
    g0 = st.glue_from_terms(t0, float(N), float(N))
    J0 = g0["KL_term"] + (gm * t0["p_m"]).sum() + (gv * t0["p_v"]).sum()
    gr0 = torch.autograd.grad(J0, [y, nz, Z, hyp])
    ref = {k: t0[k].detach() for k in ("p_m", "p_v", "recon_l", "kl_l", "ce_l")}
    ref["KL_term"] = float(g0["KL_term"])
    ref.update(zip(["dy", "dnoise", "dZ", "dhyp"], gr0))
    return ref


def run(N, M, L, seed=1234, mm_chunk=None):
    dev = torch.device("cuda")
    cfg = configs.sweep_inputs(N, M, L, device=dev, seed=seed)
    s = pkg.productSVGP(**cfg["ctor"]).to(dev)
    gm, gv = upstream(N, L, dev)
    ref = oracle(cfg, s.inducing_index_points, gm, gv)
    torch.cuda.empty_cache()

    yy = cfg["y"].clone().requires_grad_(True)
    nn = cfg["noise"].clone().requires_grad_(True)
    kw = dict(tc=True)
    if mm_chunk:
        kw["mm_chunk"] = mm_chunk
    res = s.elbo_step(cfg["aux"], yy, nn, **kw)
    gr1 = torch.autograd.grad(objective(res, gm, gv), [yy, nn, s.inducing_index_points, s._hyp()])
    out = dict(N=N, M=M, L=L, oracle="streamlined float64 on the GPU")
    for k in ("p_m", "p_v", "recon_l", "kl_l", "ce_l"):
        out[k] = rel(res[k], ref[k])
    out["KL_term"] = abs(float(res["KL_term"]) - ref["KL_term"]) / abs(ref["KL_term"])
    for name, b in zip(["dy", "dnoise", "dZ", "dhyp"], gr1):
        out[name] = rel(b, ref[name])
    return out


if __name__ == "__main__":
    N, M, L = (int(x) for x in sys.argv[1:4])
    seed = int(sys.argv[4]) if len(sys.argv) > 4 else 1234
    o = run(N, M, L, seed)
    print(json.dumps({k: (float("%.3g" % v) if isinstance(v, float) else v) for k, v in o.items()}), flush=True)
