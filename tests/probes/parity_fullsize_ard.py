"""parity_fullsize_matern.py for productSVGP with ARD length scales: the tensor-core step at (near) full size against
the streamlined float64 oracle EVALUATED ON THE GPU.

An ARD block is the isotropic factor with length scale 1 on its features divided by l_f in float64, from the same
|x|^2 + |z|^2 - 2 x.z expansion (no (N, M, d) tensor), checked against tests/ard_oracle.py on the first 256 rows.
Besides the ten usual quantities (dhyp over the whole 4 + d vector) the line reports every dhyp slot's own error,
and the slots the spec does not read (an ARD block's isotropic slot, an isotropic block's l_f) as their absolute value,
which must be exactly 0.
Usage: python tests/probes/parity_fullsize_ard.py N M L KIND_A KIND_B [seed] -> one JSON line."""
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from parity_fullsize import F64, rel, st  # noqa: E402  (also puts the repository and tests/ on sys.path)
from parity_fullsize_matern import factor64  # noqa: E402
import ard_oracle as ao  # noqa: E402
import svgp_vae_b200 as pkg  # noqa: E402
from svgp_vae_b200 import configs  # noqa: E402

# distinct per-feature length scales, geometric mean ~1 per block (the isotropic probes run at l = 1)
LS_A = [0.45, 0.8, 1.25, 2.2]
LS_B = [1.9, 0.55, 1.05, 0.9]


def kern64(X, Z, hyp, kinds, ard, same=False):
    out = None
    for i, sl in enumerate((slice(0, 4), slice(4, 8))):
        x, z = X[:, sl], Z[:, sl]
        if ard[i]:
            ls = hyp[4 + sl.start:4 + sl.stop]
            k = factor64(x / ls, z / ls, hyp[2 * i], torch.ones((), dtype=F64, device=X.device), kinds[i], same)
        else:
            k = factor64(x, z, hyp[2 * i], hyp[2 * i + 1], kinds[i], same)
        out = k if out is None else out * k
    return out


def run(N, M, L, kinds, ard=(True, True), seed=1234):
    dev = torch.device("cuda")
    cfg = configs.sweep_inputs(N, M, L, device=dev, seed=seed)
    ls = (LS_A if ard[0] else 1.0, LS_B if ard[1] else 1.0)
    s = pkg.productSVGP(**cfg["ctor"], kind_a=kinds[0], kind_b=kinds[1], length_scale=ls).to(dev)
    spec = s._spec()
    X = cfg["aux"].double()
    y = cfg["y"].double().requires_grad_(True)
    nz = cfg["noise"].double().requires_grad_(True)
    Z = s.inducing_index_points.detach().double().clone().requires_grad_(True)
    hyp = s._hyp().detach().double().clone().requires_grad_(True)
    assert rel(kern64(X[:256], Z, hyp, kinds, ard), ao.kernel_value(spec, X[:256], Z, hyp)) < 1e-12
    g = torch.Generator(device=dev).manual_seed(0)
    gm = torch.randn(N, L, generator=g, device=dev, dtype=F64)
    gv = torch.randn(N, L, generator=g, device=dev, dtype=F64)
    K_nm, K_mm = kern64(X, Z, hyp, kinds, ard), kern64(Z, Z, hyp, kinds, ard, same=True)
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
    out = dict(N=N, M=M, L=L, kinds=list(kinds), spec=list(spec), oracle="streamlined float64 on the GPU")
    for k in ("p_m", "p_v", "recon_l", "kl_l", "ce_l"):
        out[k] = rel(res[k], ref[k])
    out["KL_term"] = abs(float(res["KL_term"].detach()) - ref_KL) / abs(ref_KL)
    for name, a, b in zip(["dy", "dnoise", "dZ", "dhyp"], gr0, gr1):
        out[name] = rel(b, a)
    unread = [2 * i + 1 for i in range(2) if ard[i]] + [4 + f for f in range(8) if not ard[f // 4]]
    dh0, dh1 = gr0[3].detach().double(), gr1[3].detach().double()
    out["dhyp_slots"] = [abs(float(dh1[j])) if j in unread else abs(float(dh1[j] - dh0[j])) / abs(float(dh0[j]))
                         for j in range(dh0.numel())]
    out["dhyp_unread"] = unread
    return out


if __name__ == "__main__":
    N, M, L = (int(x) for x in sys.argv[1:4])
    kinds = (sys.argv[4], sys.argv[5])
    seed = int(sys.argv[6]) if len(sys.argv) > 6 else 1234
    o = run(N, M, L, kinds, seed=seed)
    fmt = lambda v: float("%.3g" % v) if isinstance(v, float) else ([fmt(w) for w in v] if isinstance(v, list) else v)
    print(json.dumps({k: fmt(v) for k, v in o.items()}), flush=True)
