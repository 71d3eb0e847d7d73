"""parity_fullsize_matern.py for the factor kinds the sweep does not use: linear, cosine, and a time column offset by 1e4.
The tensor-core step against the streamlined float64 oracle EVALUATED ON THE GPU.

Every factor is built in float64 from its own block: the stationary ones from per-feature differences (exact for fp32
features; the |x|^2 + |z|^2 - 2 x.z expansion of parity_fullsize.se64 subtracts terms that grow with the square of an
offset), linear and cosine from the block's dot products.  Checked against tests/matern_oracle.kernel_value on the first 256 rows.

Linear and cosine factors are low-rank, so a case is only meaningful where the oracle itself is well posed: the GATE
re-runs the oracle on K_nm and K_mm rounded to fp32 (straight through, so the gradients see the rounded values), and
that rounding must move every quantity by less than 1e-5 -- otherwise the case measures the conditioning of the problem,
not the kernels.
Usage: python tests/probes/parity_fullsize_kinds.py CASE [seed] [M] [spread] [simt] -> one JSON line (CASE of CASES; M and
the time column's spread override the case's; simt runs the SIMT step instead)."""
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from parity_fullsize import F64, st  # noqa: E402  (also puts the repository and tests/ on sys.path)
import matern_oracle as mo  # noqa: E402

QUANTITIES = ("p_m", "p_v", "recon_l", "kl_l", "ce_l", "KL_term", "dy", "dnoise", "dZ", "dhyp")
# N, M, L, the two factor kinds and block widths, the length scales, and the offset of feature 0 (a time column:
# offset + spread N(0, 1), with l = 10 on its factor).  Every case runs the tensor-core step (M >= 128; run() asserts it).
# Linear and cosine products are covered at M = 128 only (NVIDIA B200): at M = 256 lin_cos fails the gate (3.1e-5, dZ),
# cos_se fails it (1.0e-5) and se_lin passes it (1.4e-6) with the device at 9.7e-5, too close to the 1e-4 bar to keep.  The
# time column spreads over 100 length scales (spread 1000), which keeps the step well posed up to M = 1024 (gate 1.7e-6,
# device 4.9e-6).  Over 10 length scales the device missed 1e-4 at M = 1024 behind a passing gate (2.5e-4, gate 7.9e-6), and
# over one length scale already at M = 128 (1.9e-4, gate 6.1e-6) -- the SIMT step misses by the same 1.9e-4 there, so that
# gap is not in the tensor-core kernels.
CASES = {
    "lin_cos": dict(N=65536, M=128, L=4, kinds=("linear", "cosine"), dims=(16, 16), ls=(1.0, 1.0), offset=None),
    "se_lin": dict(N=65536, M=128, L=4, kinds=("se", "linear"), dims=(4, 4), ls=(1.0, 1.0), offset=None),
    "cos_se": dict(N=65536, M=128, L=4, kinds=("cosine", "se"), dims=(4, 4), ls=(1.0, 1.0), offset=None),
    "time_m32_se": dict(N=262144, M=1024, L=8, kinds=("matern32", "se"), dims=(1, 3), ls=(10.0, 1.0), offset=1e4, spread=1000.0),
}
TYPES = {"se": 1, "linear": 3, "cosine": 4, "matern12": 5, "matern32": 6, "matern52": 7}


def factor64(kind, a, b, amp, ls):
    """One factor k(a_i, b_j) in float64 from the block's own features (a: (n, d), b: (m, d))."""
    if kind in ("linear", "cosine"):
        dot = a @ b.T
        return dot if kind == "linear" else dot / (a.norm(dim=1)[:, None] * b.norm(dim=1)[None, :])
    d2 = torch.zeros((a.shape[0], b.shape[0]), dtype=a.dtype, device=a.device)
    for f in range(a.shape[1]):
        t = a[:, f:f + 1] - b[:, f][None, :]
        d2 = d2 + t * t
    if kind == "se":
        return amp * amp * torch.exp(-0.5 * d2 / (ls * ls))
    pos = d2 > 0                                     # zero gradient at r = 0, as matern_oracle.safe_norm
    r = torch.where(pos, torch.sqrt(torch.where(pos, d2, torch.ones_like(d2))), torch.zeros_like(d2))
    return mo.BY_KIND[kind](amp, ls).finish(r)


def diag64(kind, a, amp):
    """k(a_i, a_i)."""
    if kind == "linear":
        return (a * a).sum(1)
    one = torch.ones(a.shape[0], dtype=a.dtype, device=a.device)
    return one if kind == "cosine" else amp * amp * one


def kern64(X, Z, hyp, kinds, dims):
    da = dims[0]
    return (factor64(kinds[0], X[:, :da], Z[:, :da], hyp[0], hyp[1]) *
            factor64(kinds[1], X[:, da:], Z[:, da:], hyp[2], hyp[3]))


def kdiag64(X, hyp, kinds, dims):
    da = dims[0]
    return diag64(kinds[0], X[:, :da], hyp[0]) * diag64(kinds[1], X[:, da:], hyp[2])


def spec_of(kinds, dims):
    return (TYPES[kinds[0]], dims[0], TYPES[kinds[1]], dims[1])


def features(case, n, m, dev, seed):
    """Seeded features X (n, d) and inducing points Z (m, d) of a case, float32."""
    c = CASES[case]
    d = sum(c["dims"])
    X = torch.randn(n, d, generator=torch.Generator(device=dev).manual_seed(seed), device=dev)
    Z = torch.randn(m, d, generator=torch.Generator(device=dev).manual_seed(7), device=dev)
    if c["offset"] is not None:
        X[:, 0] = c["offset"] + c["spread"] * X[:, 0]
        Z[:, 0] = c["offset"] + c["spread"] * Z[:, 0]
    return X, Z


def rel(a, b):
    a, b = a.detach().double(), b.detach().double()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-300))


def oracle(X, Z0, y0, nz0, hyp0, kinds, dims, gm, gv, jitter, round_fp32=False):
    """Streamlined float64 oracle: the ten quantities (detached).  round_fp32: K_nm and K_mm rounded to fp32 (the gate)."""
    N = X.shape[0]
    X = X.double()
    y = y0.double().requires_grad_(True)
    nz = nz0.double().requires_grad_(True)
    Z = Z0.detach().double().clone().requires_grad_(True)
    hyp = hyp0.detach().double().clone().requires_grad_(True)
    K_nm, K_mm = kern64(X, Z, hyp, kinds, dims), kern64(Z, Z, hyp, kinds, dims)
    if round_fp32:
        K_nm = K_nm + (K_nm.float().double() - K_nm).detach()
        K_mm = K_mm + (K_mm.float().double() - K_mm).detach()
    t0 = st.streamlined_terms(K_nm, K_mm, kdiag64(X, hyp, kinds, dims), y, nz, float(N), jitter)
    g0 = st.glue_from_terms(t0, float(N), float(N))
    J0 = g0["KL_term"] + (gm * t0["p_m"]).sum() + (gv * t0["p_v"]).sum()
    gr = [torch.zeros_like(t) if g is None else g                # (linear x cosine: no hyper-parameter)
          for g, t in zip(torch.autograd.grad(J0, [y, nz, Z, hyp], allow_unused=True), [y, nz, Z, hyp])]
    out = {k: t0[k].detach() for k in ("p_m", "p_v", "recon_l", "kl_l", "ce_l")}
    out["KL_term"] = g0["KL_term"].detach()
    out.update(dict(zip(["dy", "dnoise", "dZ", "dhyp"], (g.detach() for g in gr))))
    return out


def compare(a, ref):
    o = {}
    for k in QUANTITIES:
        if k == "KL_term":
            o[k] = abs(float(a[k]) - float(ref[k])) / abs(float(ref[k]))
        else:
            o[k] = rel(a[k], ref[k])
    return o


def run(case, seed=1234, M=None, spread=None, tc=True):
    """tc=False runs the SIMT step on the same case (a comparison of the two paths, not a test)."""
    import svgp_vae_b200 as pkg
    from svgp_vae_b200 import backend, configs
    c = dict(CASES[case])
    if spread is not None:
        c["spread"] = spread
        CASES["_sweep"] = c
        case = "_sweep"
    N, L, kinds, dims = c["N"], c["L"], c["kinds"], c["dims"]
    M = c["M"] if M is None else M
    dev = torch.device("cuda")
    cfg = configs.sweep_inputs(N, M, L, device=dev, seed=seed)
    X, Z0 = features(case, N, M, dev, seed)
    if tc:
        assert backend.get_backend().want_tc(N, M), "not a tensor-core size: the step would run the SIMT kernels"
    s = pkg.productSVGP(Z0.cpu().numpy(), dim_a=dims[0], dim_b=dims[1], jitter=cfg["ctor"]["jitter"], N_train=N, L=L,
                        kind_a=kinds[0], kind_b=kinds[1], length_scale=c["ls"]).to(dev)
    hyp = s._hyp().detach()
    Xd = X.double()
    assert rel(kern64(Xd[:256], Z0.double(), hyp.double(), kinds, dims),
               mo.kernel_value(spec_of(kinds, dims), X[:256], Z0, hyp)) < 1e-12
    gm = torch.randn(N, L, generator=torch.Generator(device=dev).manual_seed(0), device=dev, dtype=F64)
    gv = torch.randn(N, L, generator=torch.Generator(device=dev).manual_seed(1), device=dev, dtype=F64)
    ref = oracle(X, Z0, cfg["y"], cfg["noise"], hyp, kinds, dims, gm, gv, s.jitter)
    torch.cuda.empty_cache()
    gate = compare(oracle(X, Z0, cfg["y"], cfg["noise"], hyp, kinds, dims, gm, gv, s.jitter, round_fp32=True), ref)
    torch.cuda.empty_cache()

    yy = cfg["y"].clone().requires_grad_(True)
    nn = cfg["noise"].clone().requires_grad_(True)
    res = s.elbo_step(X, yy, nn, tc=tc)
    J1 = res["KL_term"] + (gm.float() * res["p_m"]).sum().double() + (gv.float() * res["p_v"]).sum().double()
    gr1 = torch.autograd.grad(J1, [yy, nn, s.inducing_index_points, s._hyp()])
    dev_out = {k: res[k] for k in ("p_m", "p_v", "recon_l", "kl_l", "ce_l", "KL_term")}
    dev_out.update(dict(zip(["dy", "dnoise", "dZ", "dhyp"], gr1)))
    out = dict(case=case, N=N, M=M, L=L, kinds=list(kinds), dims=list(dims), offset=c["offset"], spread=c.get("spread"),
               path="tensor-core" if tc else "simt", oracle="streamlined float64 on the GPU")
    out.update(compare(dev_out, ref))
    out["gate"] = gate
    out["max"] = max(out[k] for k in QUANTITIES)
    out["gate_max"] = max(gate.values())
    return out


if __name__ == "__main__":
    case = sys.argv[1]
    seed = int(sys.argv[2]) if len(sys.argv) > 2 else 1234
    a = sys.argv
    o = run(case, seed, int(a[3]) if len(a) > 3 and a[3] != "-" else None, float(a[4]) if len(a) > 4 and a[4] != "-" else None,
            tc=not (len(a) > 5 and a[5] == "simt"))
    fmt = lambda v: float("%.3g" % v) if isinstance(v, float) else v
    print(json.dumps({k: ({kk: fmt(vv) for kk, vv in v.items()} if isinstance(v, dict) else fmt(v)) for k, v in o.items()}),
          flush=True)
