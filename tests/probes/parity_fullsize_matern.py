"""parity_fullsize.py for productSVGP with Matern factors: the tensor-core step at (near) full size against the
streamlined float64 oracle EVALUATED ON THE GPU.

Each factor is restated in float64 from the same |x|^2 + |z|^2 - 2 x.z expansion as parity_fullsize.se64 (so that no
(N, M, d) tensor is needed) and checked against tests/matern_oracle.py on the first 256 rows.
Usage: python tests/probes/parity_fullsize_matern.py N M L KIND_A KIND_B [seed] -> one JSON line."""
import json
import math
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from parity_fullsize import F64, rel, se64, st  # noqa: E402  (also puts the repository and tests/ on sys.path)
import matern_oracle as mo  # noqa: E402
import svgp_vae_b200 as pkg  # noqa: E402
from svgp_vae_b200 import configs  # noqa: E402
from oracle import tfp_kernels as tfk  # noqa: E402

_C = {"matern12": 1.0, "matern32": math.sqrt(3.0), "matern52": math.sqrt(5.0)}


def matern64(a, b, amp, ls, kind, same=False):
    """Matern factor from the expansion.  same=True (K_mm): the diagonal distance is set to exactly 0 -- the expansion
    leaves ~1e-16 there, whose square root would put a spurious 1 / r into the Matern 1/2 gradient; r = 0 takes the zero
    (sub)gradient, as in matern_oracle."""
    d2 = ((a * a).sum(1)[:, None] + (b * b).sum(1)[None, :] - 2.0 * (a @ b.T)).clamp_min(0.0)
    if same:
        d2 = d2.masked_fill(torch.eye(d2.shape[0], dtype=torch.bool, device=d2.device), 0.0)
    pos = d2 > 0
    r = torch.where(pos, torch.sqrt(torch.where(pos, d2, torch.ones_like(d2))), torch.zeros_like(d2))
    return mo.BY_KIND[kind](amp, ls).finish(r)


def factor64(a, b, amp, ls, kind, same=False):
    return se64(a, b, amp, ls) if kind == "se" else matern64(a, b, amp, ls, kind, same)


def kern64(X, Z, hyp, kinds, same=False):
    return factor64(X[:, :4], Z[:, :4], hyp[0], hyp[1], kinds[0], same) * factor64(X[:, 4:], Z[:, 4:], hyp[2], hyp[3], kinds[1], same)


def run(N, M, L, kinds, seed=1234):
    dev = torch.device("cuda")
    cfg = configs.sweep_inputs(N, M, L, device=dev, seed=seed)
    s = pkg.productSVGP(**cfg["ctor"], kind_a=kinds[0], kind_b=kinds[1]).to(dev)
    X = cfg["aux"].double()
    y = cfg["y"].double().requires_grad_(True)
    nz = cfg["noise"].double().requires_grad_(True)
    Z = s.inducing_index_points.detach().double().clone().requires_grad_(True)
    hyp = torch.ones(4, dtype=F64, device=dev, requires_grad=True)
    one = torch.ones((), dtype=F64, device=dev)
    ref_cls = lambda kind: tfk.ExponentiatedQuadratic if kind == "se" else mo.BY_KIND[kind]
    ref_k = ref_cls(kinds[0])(one, one).matrix(X[:256, :4], Z[:, :4]) * ref_cls(kinds[1])(one, one).matrix(X[:256, 4:], Z[:, 4:])
    assert rel(kern64(X[:256], Z, hyp, kinds), ref_k) < 1e-12
    g = torch.Generator(device=dev).manual_seed(0)
    gm = torch.randn(N, L, generator=g, device=dev, dtype=F64)
    gv = torch.randn(N, L, generator=g, device=dev, dtype=F64)
    K_nm, K_mm = kern64(X, Z, hyp, kinds), kern64(Z, Z, hyp, kinds, same=True)
    kappa = (hyp[0] * hyp[2]) ** 2 * torch.ones(N, dtype=F64, device=dev)
    t0 = st.streamlined_terms(K_nm, K_mm, kappa, y, nz, float(N), cfg["ctor"]["jitter"])
    g0 = st.glue_from_terms(t0, float(N), float(N))
    J0 = g0["KL_term"] + (gm * t0["p_m"]).sum() + (gv * t0["p_v"]).sum()
    gr0 = torch.autograd.grad(J0, [y, nz, Z, hyp])
    ref = {k: t0[k].detach() for k in ("p_m", "p_v", "recon_l", "kl_l", "ce_l")}
    ref_KL = float(g0["KL_term"].detach())
    del t0, g0, J0, K_nm, K_mm
    torch.cuda.empty_cache()

    yy = cfg["y"].clone().requires_grad_(True)
    nn = cfg["noise"].clone().requires_grad_(True)
    res = s.elbo_step(cfg["aux"], yy, nn, tc=True)
    J1 = res["KL_term"] + (gm.float() * res["p_m"]).sum().double() + (gv.float() * res["p_v"]).sum().double()
    gr1 = torch.autograd.grad(J1, [yy, nn, s.inducing_index_points, s._hyp()])
    out = dict(N=N, M=M, L=L, kinds=list(kinds), oracle="streamlined float64 on the GPU")
    for k in ("p_m", "p_v", "recon_l", "kl_l", "ce_l"):
        out[k] = rel(res[k], ref[k])
    out["KL_term"] = abs(float(res["KL_term"].detach()) - ref_KL) / abs(ref_KL)
    for name, a, b in zip(["dy", "dnoise", "dZ", "dhyp"], gr0, gr1):
        out[name] = rel(b, a)
    return out


if __name__ == "__main__":
    N, M, L = (int(x) for x in sys.argv[1:4])
    kinds = (sys.argv[4], sys.argv[5])
    seed = int(sys.argv[6]) if len(sys.argv) > 6 else 1234
    o = run(N, M, L, kinds, seed)
    print(json.dumps({k: (float("%.3g" % v) if isinstance(v, float) else v) for k, v in o.items()}), flush=True)
