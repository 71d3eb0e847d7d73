"""What ARD length scales cost on the bench workload: SE x SE against SE|ARD x SE|ARD productSVGP (N = 1e6, M = 1024,
L = 64, [4 | 4] features).  K1 forward (svgp_kernel_fwd_i8, the integer tensor-core operand builder of the step), K1
backward (svgp_kernel_bwd, the Z pass the step runs on K_nm) and one whole step (elbo_step forward + backward of
J = KL_term + <g_m, p_m> + <g_v, p_v>, as bench.py).  The two arms alternate inside one process, each warmed up, timed
with CUDA events; the isotropic arm is the baseline of the same call.  A separate torch.profiler pass then lists the
K1 kernels each arm's step launches: the ARD arm has to stay on the SE44 kernels (kernel_fwd_i8_kernel<true, *> and
kernel_bwd_z_se44_kernel).  Prints one JSON line (and writes it to --out).

    python tools/ard_k1_timing.py [--n N] [--reps R] [--out FILE]
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
from svgp_vae_b200 import backend, configs  # noqa: E402
from matern_k1_timing import card, event_time  # noqa: E402

# distinct per-feature length scales, geometric mean ~1 per block (the isotropic arm runs at l = 1)
ARMS = {"se_se": (1.0, 1.0), "se_se_ard": ([0.45, 0.8, 1.25, 2.2], [1.9, 0.55, 1.05, 0.9])}
K1_NAMES = ("kernel_fwd_i8_kernel", "kernel_bwd_z_se44_kernel", "kernel_bwd_kernel", "kernel_fwd_kernel",
            "kernel_fwd_planes_kernel", "kernel_fwd_f64_kernel", "kernel_diag")


def k1_kernels(step):
    """Names (demangled, arguments dropped) and call counts of the K1 kernels one step launches."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        step()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        if any(k in e.key for k in K1_NAMES):
            out[e.key.split("(")[0].replace("void ", "")] = e.count
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1_000_000)
    ap.add_argument("--m", type=int, default=1024)
    ap.add_argument("--l", type=int, default=64)
    ap.add_argument("--reps", type=int, default=5, help="alternations of the two arms")
    ap.add_argument("--out")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "a timing needs the GPU"
    dev = torch.device("cuda")
    be = backend.get_backend()
    N, M, L = args.n, args.m, args.l
    cfg = configs.sweep_inputs(N, M, L, device=dev)
    aux, y, noise = cfg["aux"], cfg["y"], cfg["noise"]
    g = torch.Generator(device=dev).manual_seed(99)
    gm, gv = torch.randn(N, L, generator=g, device=dev), torch.randn(N, L, generator=g, device=dev)
    G = torch.randn(N, M, generator=g, device=dev) * 1e-3          # cotangent of K_nm for the backward alone
    Fz = torch.from_numpy(cfg["ctor"]["initial_inducing_points"]).float().to(dev)

    fns, specs = {}, {}
    for arm, ls in ARMS.items():
        s = pkg.productSVGP(**cfg["ctor"], length_scale=ls).to(dev)
        spec, hyp = s._spec(), s._hyp().detach().float().contiguous()
        specs[arm] = list(spec)

        def step(s=s):
            yy, nn = y.clone().requires_grad_(True), noise.clone().requires_grad_(True)
            for p in s.parameters():
                p.grad = None
            res = s.elbo_step(aux, yy, nn, return_A_hat=False)
            J = (gm * res["p_m"]).sum().double() + (gv * res["p_v"]).sum().double() + res["KL_term"]
            J.backward()

        fns[arm] = dict(
            k1_fwd=lambda spec=spec, hyp=hyp: be.kernel_fwd(spec, aux, Fz, hyp, tc=True, i8=True),
            k1_bwd=lambda spec=spec, hyp=hyp: be.kernel_bwd(spec, aux, Fz, hyp, G, need_x=False, need_z=True),
            step=step)

    kinds_timed = ("k1_fwd", "k1_bwd", "step")
    reps_of = dict(k1_fwd=10, k1_bwd=5, step=1)
    for arm in ARMS:                                                    # warm-up: every shape and module of both arms
        for k in kinds_timed:
            for _ in range(2):
                fns[arm][k]()
    torch.cuda.synchronize()
    times = {arm: {k: [] for k in kinds_timed} for arm in ARMS}
    for _ in range(args.reps):
        for arm in ARMS:
            for k in kinds_timed:
                times[arm][k].append(event_time(fns[arm][k], reps_of[k]))

    out = dict(what="SE|ARD x SE|ARD vs SE x SE, productSVGP [4|4]", N=N, M=M, L=L, reps=args.reps,
               card=card(), torch=torch.__version__, unit="ms", specs=specs)
    for arm in ARMS:
        out[arm] = {k: dict(median=round(statistics.median(v), 3), min=round(min(v), 3), max=round(max(v), 3))
                    for k, v in times[arm].items()}
    out["ratio_ard_over_iso"] = {k: round(out["se_se_ard"][k]["median"] / out["se_se"][k]["median"], 3) for k in kinds_timed}
    out["k1_share_of_step"] = {arm: round((out[arm]["k1_fwd"]["median"] + out[arm]["k1_bwd"]["median"])
                                          / out[arm]["step"]["median"], 3) for arm in ARMS}
    out["k1_kernels_of_step"] = {arm: k1_kernels(fns[arm]["step"]) for arm in ARMS}      # profiled after the timing
    line = json.dumps(out)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
