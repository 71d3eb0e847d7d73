"""What summing the per-entry differences c (x_f - z_f) in the K1 Z pass costs on the bench workload (productSVGP SE x SE
on [4 | 4], N = 1e6, M = 1024, L = 64): the SE44 Z pass (svgp_kernel_bwd with dFz only, kernel_bwd_z_se44_kernel) and
one whole step (elbo_step forward + backward of J = KL_term + <g_m, p_m> + <g_v, p_v>, as bench.py), and the Z pass of the
generic kernel (kernel_bwd_kernel) for the specs in GENERIC on N(0, 1) features of the same N and M, for the in-tree
library against a baseline library built from another revision of the same sources (--baseline-lib).  The two arms
alternate inside one process, each warmed up, timed with CUDA events; medians of --reps.  Both arms also report the
largest relative difference of their dz from the other arm's.  Prints one JSON line (and writes it to --out).

    python tools/k1_z_diff_timing.py --baseline-lib PATH [--n N] [--reps R] [--out FILE]
"""
import argparse
import json
import os
import statistics
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import svgp_vae_b200 as pkg  # noqa: E402
from svgp_vae_b200 import _lib, backend, configs  # noqa: E402
from matern_k1_timing import card, event_time  # noqa: E402


# generic Z-pass specs: SPRITES' SE on [8 | 16], SE|ARD x SE off [4 | 4], Matern 5/2 (double partials before and after),
# EXPSIN x LINEAR (MNIST), linear x cosine on [16 | 16] (fails on a library without the shared-memory opt-in: reported as such)
GENERIC = {"se_8_16": ((1, 8, 1, 16), [1.0, 1.3, 1.0, 0.8]),
           "se_ard_3_2": ((17, 3, 1, 2), [1.0, 1.0, 1.0, 0.8, 0.7, 0.85, 1.0, 1.0, 1.0]),
           "m52_m52": ((7, 4, 7, 4), [1.0, 1.3, 1.0, 0.8]),
           "expsin_linear": ((2, 1, 3, 8), [1.0, 1.3, 1.0, 1.0]),
           "linear_cosine_16_16": ((3, 16, 4, 16), [1.0, 1.0, 1.0, 1.0])}


def load_library(path):
    """A second copy of the C ABI from another build (ctypes keeps the two apart); _lib.load() itself is left as it was."""
    saved = _lib.LIB_PATH, _lib._lib
    _lib.LIB_PATH, _lib._lib = path, None
    try:
        return _lib.load()
    finally:
        _lib.LIB_PATH, _lib._lib = saved


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--baseline-lib", required=True, help="libsvgp_b200.so built from the baseline revision")
    ap.add_argument("--n", type=int, default=1_000_000)
    ap.add_argument("--m", type=int, default=1024)
    ap.add_argument("--l", type=int, default=64)
    ap.add_argument("--reps", type=int, default=5, help="alternations of the two arms")
    ap.add_argument("--out")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "a timing needs the GPU"
    dev = torch.device("cuda")
    libs = {"baseline": load_library(os.path.abspath(args.baseline_lib)), "change": load_library(_lib.LIB_PATH)}
    be = backend.get_backend()
    N, M, L = args.n, args.m, args.l
    cfg = configs.sweep_inputs(N, M, L, device=dev)
    aux, y, noise = cfg["aux"], cfg["y"], cfg["noise"]
    g = torch.Generator(device=dev).manual_seed(99)
    gm, gv = torch.randn(N, L, generator=g, device=dev), torch.randn(N, L, generator=g, device=dev)
    G = torch.randn(N, M, generator=g, device=dev) * 1e-3          # cotangent of K_nm for the Z pass alone
    Fz = torch.from_numpy(cfg["ctor"]["initial_inducing_points"]).float().to(dev)
    s = pkg.productSVGP(**cfg["ctor"]).to(dev)
    spec, hyp = s._spec(), s._hyp().detach().float().contiguous()

    def step():
        yy, nn = y.clone().requires_grad_(True), noise.clone().requires_grad_(True)
        for p in s.parameters():
            p.grad = None
        res = s.elbo_step(aux, yy, nn, return_A_hat=False)
        J = (gm * res["p_m"]).sum().double() + (gv * res["p_v"]).sum().double() + res["KL_term"]
        J.backward()

    fns = dict(k1_bwd_z=lambda: be.kernel_bwd(spec, aux, Fz, hyp, G, need_x=False, need_z=True), step=step)
    reps_of = dict(k1_bwd_z=5, step=1)
    for name, (gspec, ghyp) in GENERIC.items():
        d = gspec[1] + gspec[3]
        Xg = torch.randn(N, d, generator=g, device=dev)
        Zg = torch.randn(M, d, generator=g, device=dev)
        hg = torch.tensor(ghyp, device=dev)
        fns["z_" + name] = lambda gspec=gspec, Xg=Xg, Zg=Zg, hg=hg: be.kernel_bwd(gspec, Xg, Zg, hg, G, need_x=False, need_z=True)
        reps_of["z_" + name] = 2
    dz, failed = {}, {}
    for arm, lib in libs.items():                                      # warm-up: every shape and module of both arms
        _lib._lib = lib
        for k in list(fns):
            try:
                for _ in range(2):
                    fns[k]()
            except _lib.SvgpLibraryError as e:
                failed.setdefault(arm, {})[k] = str(e)
        dz[arm] = fns["k1_bwd_z"]()[1]
    # a call that fails on either arm is reported, not timed
    for k in {k for f in failed.values() for k in f}:
        fns.pop(k)
    torch.cuda.synchronize()
    times = {arm: {k: [] for k in fns} for arm in libs}
    for _ in range(args.reps):
        for arm, lib in libs.items():
            _lib._lib = lib
            for k in fns:
                times[arm][k].append(event_time(fns[k], reps_of[k]))
    _lib._lib = libs["change"]

    out = dict(what="K1 Z pass on per-entry differences: in-tree library vs baseline, productSVGP SE x SE [4|4]",
               N=N, M=M, L=L, reps=args.reps, card=card(), torch=torch.__version__, unit="ms", spec=list(spec),
               dz_rel_diff=float((dz["change"] - dz["baseline"]).abs().max() / dz["baseline"].abs().max()),
               generic_specs={k: list(v[0]) for k, v in GENERIC.items()}, failed=failed)
    for arm in libs:
        out[arm] = {k: dict(median=round(statistics.median(v), 3), min=round(min(v), 3), max=round(max(v), 3))
                    for k, v in times[arm].items()}
    out["ratio_change_over_baseline"] = {k: round(out["change"][k]["median"] / out["baseline"][k]["median"], 3) for k in fns}
    line = json.dumps(out)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
