#!/usr/bin/env python
"""Benchmark of the SVGP ELBO + gradient step (BASELINE.json metric) on N GPUs of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's CUDA path
    python bench.py --impl reference [--steps K] [--warmup W]      # CPU restatement of the reference path
    python bench.py --steps K --dump-outputs DIR                   # + the last timed step's outputs as DIR/<name>.npy

One step = forward (p_m, p_v, inside_elbo_recon/kl, ce_term) + backward of
J = KL_term + <g_m, p_m> + <g_v, p_v> to y, noise, inducing points and kernel hypers, on the SWEEP
workload of SURVEY 8(d): N = 1e6 datapoints per GPU (weak scaling; --strong splits N over the GPUs), M = 1024,
L = 64, product-SE kernel d = 4 + 4, jitter 1e-2.  Prints ONE JSON line (rank 0).  `value` is device-resident
throughput; `e2e` includes the pinned-host -> device copy of (aux, y, noise) and the device -> host read of
p_m, p_v, dy, dnoise and the scalars every step.  roofline: tensor-core bound; the integer tensor-core path issues
10 tcgen05 kind::i8 MMAs per algorithmic MAC at twice the bf16 rate (= 5 bf16-equivalents; the fp16-split row quads
issue 3); peak = the driver-measured sustained bf16/fp16 dense GEMM rate of MEASURED_PEAKS.json (an fp16 cuBLAS GEMM
is also timed in-run).  --impl reference: the CPU restatement of the reference path on the host cores.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

# torchrun exports OMP_NUM_THREADS=1 to every worker; the reference arm is a CPU run that should use all host threads
# (rank 0 alone does any work there), so drop that default before torch / MKL read it
if "reference" in sys.argv and os.environ.get("OMP_NUM_THREADS") == "1" and "RANK" in os.environ:
    del os.environ["OMP_NUM_THREADS"]

import torch  # noqa: E402

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_PER_GPU, M_IND, L_CH = 1_000_000, 1024, 64
METRIC = "SVGP ELBO+grad datapoints/s at M=1024,L=64"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    # (--rows / --inducing / --channels: spellings that torchrun's own option abbreviations do not swallow)
    ap.add_argument("--n", "--rows", dest="n", type=int, default=N_PER_GPU, help="datapoints per GPU (default: the named workload)")
    ap.add_argument("--m", "--inducing", dest="m", type=int, default=M_IND)
    ap.add_argument("--l", "--channels", dest="l", type=int, default=L_CH)
    ap.add_argument("--mm-chunk", type=int, default=0, help="channels per chunk of the float64 M x M stage (0 = automatic)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--lean", action="store_true", help="big configurations on a GPU budget: no extra profiling step (the per-kernel / collective "
                    "profile is taken on the last timed step's twin run only when not lean: here on the first warm-up step) and no e2e loop")
    ap.add_argument("--strong", action="store_true", help="strong scaling: --n is the TOTAL number of datapoints, split over the GPUs")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one returned (p_m, p_v, the "
                    "ELBO terms, mu_hat, A_hat, the gradients of y, noise and the parameters) to DIR/<name>.npy; large arrays are "
                    "cut to fixed, seeded samples so that the dump stays below 64 MB (rank 0's rows on several GPUs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


# --------------------------------------------------------------------------------------------------
# clocks
# --------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.samples, self.stop = index, [], threading.Event()
        self.thread = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        while not self.stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in out.strip().split(",")]
                if len(f) >= 6:
                    self.samples.append(f)
            except Exception:  # noqa: BLE001
                pass
            self.stop.wait(0.2)

    def __enter__(self):
        self.thread.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.thread.join(timeout=6)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = sorted(int(s[0]) for s in self.samples if s[0].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(s[2 + i].lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": int(self.samples[0][1]) if self.samples[0][1].isdigit() else None,
                "reasons": reasons, "samples": len(self.samples)}


# --------------------------------------------------------------------------------------------------
# CPU restatement (the "reference arm" and the cpu_baseline leg): oracle/ is only touched here
# --------------------------------------------------------------------------------------------------
def workload_name(args, world):
    """The one workload string both arms print (the driver compares the `config` of the two lines)."""
    which = "configs[4] shapes" if (args.m, args.l) == (4096, 128) else "configs[3]"
    return "SWEEP N=%d per GPU x %d GPU(s), M=%d, L=%d, product-SE d=4+4, jitter 1e-2 (%s)" % (args.n, world, args.m, args.l, which)


def workload_config(args, world):
    """The `config` object of the JSON line: identical for both arms (it describes the workload, not an implementation)."""
    strong = getattr(args, "strong", False)
    n_gpu = args.n // world if strong else args.n
    name = workload_name(args, world) if not strong else (
        "SWEEP N=%d TOTAL split over %d GPU(s), M=%d, L=%d, product-SE d=4+4, jitter 1e-2 (configs[3], strong scaling)" % (args.n, world, args.m, args.l))
    return {"workload": name,
            "l2": "inputs_exceed_l2 (K_nm alone is N x M x 4 B = %.1f GB per GPU, re-streamed by every pass of the step)" % (4.0 * n_gpu * args.m / 1e9),
            "parallelism": "datapoints sharded over %d GPU(s)" % world}


def cpu_reference_timer(max_rows, M, L):
    """-> full(rows): seconds of one fwd + bwd of the streamlined float64 restatement on `rows` rows of the workload."""
    from oracle import svgp_streamlined as st
    from oracle import tfp_kernels as tfk
    from svgp_vae_b200 import configs
    cfg = configs.sweep_inputs(max_rows, M, L, device="cpu", N_train=max_rows)
    X, y, nz = cfg["aux"].double(), cfg["y"].double().requires_grad_(True), cfg["noise"].double().requires_grad_(True)
    Z = torch.as_tensor(cfg["ctor"]["initial_inducing_points"]).double().requires_grad_(True)
    one = torch.ones((), dtype=torch.float64)
    kern = lambda a, b: tfk.ExponentiatedQuadratic(one, one).matrix(a[:, :4], b[:, :4]) * tfk.ExponentiatedQuadratic(one, one).matrix(a[:, 4:], b[:, 4:])
    g = torch.Generator().manual_seed(0)
    gm, gv = torch.randn(max_rows, L, generator=g, dtype=torch.float64), torch.randn(max_rows, L, generator=g, dtype=torch.float64)

    def full(rows):
        t0 = time.perf_counter()
        K_nm, K_mm = kern(X[:rows], Z), kern(Z, Z)
        kappa = torch.ones(rows, dtype=torch.float64)
        t = st.streamlined_terms(K_nm, K_mm, kappa, y[:rows], nz[:rows], float(rows), 1e-2)
        gl = st.glue_from_terms(t, float(rows), float(rows))
        J = gl["KL_term"] + (gm[:rows] * t["p_m"]).sum() + (gv[:rows] * t["p_v"]).sum()
        torch.autograd.grad(J, [y, nz, Z])
        return time.perf_counter() - t0
    return full


def fit_rows(samples):
    """Least-squares line t = intercept + slope * rows through (rows, seconds) samples -> (slope, intercept, max relative residual).
    The step costs a row-independent float64 M x M part (intercept) plus a part proportional to the datapoints (slope)."""
    n = len(samples)
    mx = sum(r for r, _ in samples) / n
    my = sum(t for _, t in samples) / n
    sxx = sum((r - mx) ** 2 for r, _ in samples)
    if sxx == 0:                       # one size only: no separation possible, charge everything to the rows (pessimistic for the CPU)
        return my / mx, 0.0, None
    slope = sum((r - mx) * (t - my) for r, t in samples) / sxx
    slope = max(slope, 1e-12)
    icpt = max(my - slope * mx, 0.0)
    resid = max(abs(icpt + slope * r - t) / t for r, t in samples)
    return slope, icpt, resid


def literal_small_configs():
    """fwd + bwd of the LITERAL restatement (per-channel loop, explicit inverses, the (b, m, m) tensor: what the reference's
    graph does) on the reference's own shapes, median of 3 -- BASELINE.md section 4."""
    out = {}
    try:
        from oracle import svgp_literal as lit
        from svgp_vae_b200 import configs
        fix = os.path.join(ROOT, "tests", "golden", "mnist_aux.npz")
        cases = {"mnist_b256_m32_L16": ("mnist", configs.mnist_inputs(fix, L=16)), "sprites_b500_M72_L64": ("sprites", configs.sprites_inputs(M=72, L=64))}
        for name, (kind, cfg) in cases.items():
            o = (lit.MnistSVGP if kind == "mnist" else lit.SpritesSVGP)(name="o", **cfg["ctor"])
            ts = []
            for _ in range(3):
                y = cfg["y"].double().clone().requires_grad_(True)
                nz = cfg["noise"].double().clone().requires_grad_(True)
                t0 = time.perf_counter()
                res = lit.minibatch_glue(o, cfg["aux"].double(), y, nz, clip_pv=(kind == "sprites"))
                torch.autograd.grad(res["KL_term"] + res["p_m"].sum() + res["p_v"].sum(), [y, nz])
                ts.append(time.perf_counter() - t0)
            out[name] = {"ms_per_step": 1e3 * sorted(ts)[1], "datapoints_per_s": cfg["aux"].shape[0] / sorted(ts)[1]}
    except Exception as e:  # noqa: BLE001
        out["error"] = repr(e)
    return out


def cpu_baseline(args, n_total):
    """The cpu_baseline leg of the GPU arm (rank 0, one GPU): two sizes, ~10-30 s of CPU work on a many-core host."""
    threads = torch.get_num_threads()     # (torch.set_num_threads breaks MKL's batched LU in this image: leave the default)
    full = cpu_reference_timer(4096, args.m, args.l)
    full(256)                             # warm-up (thread pools, allocator)
    samples = [(r, full(r)) for r in (1024, 4096)]
    slope, icpt, resid = fit_rows(samples)
    t_total = slope * n_total + icpt
    return {"value": n_total / t_total, "unit": "datapoints/s", "cores": threads, "kind": "port", "extrapolated": True,
            "sample_rows": [r for r, _ in samples], "sample_seconds": [round(t, 3) for _, t in samples],
            "fit": {"seconds_per_row": slope, "row_independent_seconds": icpt},
            "sample": "streamlined float64 restatement (oracle/svgp_streamlined.py, torch-CPU/MKL, %d threads; TensorFlow 1.15 is not installable) "
                      "fwd+bwd on 1024 and 4096 rows of the same workload (M=%d, L=%d); t = %.2f s + %.3g s/row extrapolated linearly in "
                      "rows to N=%d" % (threads, args.m, args.l, icpt, slope, n_total),
            "literal_small_configs": literal_small_configs()}


def run_reference(args):
    """Reference arm: the CPU restatement of the reference path on the host cores.  Each step = one fwd + bwd on a bounded
    sample of the workload (sizes cycle through 8192 / 2048 / 4096 rows so that the row-proportional cost and the
    row-independent M x M cost separate by a line fit over the timed steps); the whole run is time-boxed."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = torch.get_num_threads()
    n_total = args.n if args.strong else args.n * args.gpus
    sizes = [8192, 2048, 4096]
    full = cpu_reference_timer(max(sizes), args.m, args.l)
    t_start = time.perf_counter()
    for _ in range(max(1, min(args.warmup, 2))):
        full(512)                                               # untimed warm-up steps (small: the budget goes to the timed ones)
    samples = []
    for i in range(max(args.steps, 3)):
        samples.append((sizes[i % 3], full(sizes[i % 3])))
        if len(samples) >= 3 and time.perf_counter() - t_start > 200:      # keep the whole run within minutes
            break
    slope, icpt, resid = fit_rows(samples)
    # spread of the row cost over the repeats of the largest size (the extrapolation's dominant term)
    big = sorted(t for r, t in samples if r == sizes[0])
    t_total = slope * n_total + icpt
    value = n_total / t_total
    world = args.gpus
    cb = {"value": value, "unit": "datapoints/s", "cores": threads, "kind": "port", "extrapolated": True,
          "sample_rows": [r for r, _ in samples], "sample_seconds": [round(t, 3) for _, t in samples],
          "fit": {"seconds_per_row": slope, "row_independent_seconds": icpt, "max_rel_residual": resid,
                  "largest_size_seconds_min_max": [big[0], big[-1]] if big else None},
          "sample": "each step = fwd+bwd of the streamlined float64 restatement (oracle/svgp_streamlined.py, torch-CPU/MKL, %d threads) on "
                    "8192 / 2048 / 4096 rows in turn; line fit t = %.2f s + %.3g s/row over %d timed steps, extrapolated linearly in rows to "
                    "N=%d; TensorFlow 1.15 / TFP 0.8 cannot be installed here" % (threads, icpt, slope, len(samples), n_total)}
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "datapoints/s", "n_gpus": args.gpus, "steps": len(samples),
            "warmup": args.warmup, "ms_per_step": 1e3 * t_total, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "extrapolated": True,
            "config": workload_config(args, world),
            "cpu_baseline": cb,
            "e2e": {"value": value, "unit": "datapoints/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------------------
def measure_f16_peak(dev):
    old = torch.backends.cuda.matmul.allow_tf32
    n = 8192
    a = torch.randn(n, n, device=dev).half()
    b = torch.randn(n, n, device=dev).half()
    for _ in range(3):
        a @ b
    torch.cuda.synchronize()
    best = 0.0
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        a @ b
        e1.record()
        torch.cuda.synchronize()
        best = max(best, 2 * n ** 3 / (e0.elapsed_time(e1) * 1e-3) / 1e12)
    torch.backends.cuda.matmul.allow_tf32 = old
    del a, b
    return best


DUMP_BYTES = 48 << 20                 # array data of --dump-outputs: the files, headers included, stay well below 64 MB
DUMP_WHOLE_BYTES = 1 << 20            # arrays up to this size are always written whole


def dump_outputs(out_dir, arrays, n_rows):
    """Write each tensor of `arrays` to out_dir/<name>.npy, float64 ones as float64 and all others as float32, at most
    DUMP_BYTES of array data in all.  Arrays of up to DUMP_WHOLE_BYTES are written whole; when the others do not fit in
    what is left, each of them keeps the same fraction of itself: arrays with one row per datapoint a sample of rows
    (seed 0, ascending, the same rows for all of them), any other array a sample of its flattened elements (seed 0,
    ascending).  The samples depend only on the shapes, so two builds run with the same arguments can be compared array
    for array."""
    import numpy as np
    arrays = {k: v.detach() if v.dtype == torch.float64 else v.detach().float() for k, v in arrays.items()}
    nbytes = lambda v: v.numel() * v.element_size()
    large = {k for k, v in arrays.items() if nbytes(v) > DUMP_WHOLE_BYTES}
    room = DUMP_BYTES - sum(nbytes(v) for k, v in arrays.items() if k not in large)
    frac = min(1.0, room / max(1, sum(nbytes(arrays[k]) for k in large)))
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        if k in large and frac < 1.0:
            g = torch.Generator().manual_seed(0)
            if v.shape[0] == n_rows:
                idx = torch.randperm(n_rows, generator=g)[:int(n_rows * frac)].sort().values
                v = v.index_select(0, idx.to(v.device))
            else:
                idx = torch.randint(v.numel(), (int(v.numel() * frac),), generator=g).unique()     # sorted, at most that many
                v = v.reshape(-1).index_select(0, idx.to(v.device))
        np.save(os.path.join(out_dir, k + ".npy"), v.cpu().numpy())


def run_gpu(args):
    import torch.distributed as dist
    import svgp_vae_b200 as pkg
    from svgp_vae_b200 import backend, configs
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    group = None
    if world > 1:
        # NCCL prints its version banner on stdout when the first communicator comes up: keep stdout for the ONE JSON line
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            group = dist.group.WORLD
            dist.all_reduce(torch.zeros(1, device=dev), group=group)
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    be = backend.get_backend()
    N, M, L = args.n, args.m, args.l
    if args.strong:                                # configs[3] read as a strong-scaling sweep: the N = 1e6 problem split over the ranks
        N = (args.n + world - 1) // world
    n_total = N * world

    cfg = configs.sweep_inputs(N, M, L, device=dev, rank=rank, N_train=n_total)
    svgp = pkg.productSVGP(**cfg["ctor"]).to(dev)
    aux, y, noise = cfg["aux"], cfg["y"], cfg["noise"]
    g = torch.Generator(device=dev).manual_seed(99 + rank)
    gm = torch.randn(N, L, generator=g, device=dev)
    gv = torch.randn(N, L, generator=g, device=dev)
    params = [p for p in svgp.parameters()]

    def step(aux_d, y_d, nz_d):
        y_d.requires_grad_(True); nz_d.requires_grad_(True)
        for p in params:
            p.grad = None
        res = svgp.elbo_step(aux_d, y_d, nz_d, group=group, mm_chunk=args.mm_chunk or None, return_A_hat=False)
        # per-rank loss = local decoder stand-in + this rank's share of the replicated global scalar
        J = (gm * res["p_m"]).sum().double() + (gv * res["p_v"]).sum().double() + res["KL_term"] / world
        J.backward()
        if group is not None:                                    # replicated parameters: sum the per-rank partial gradients
            flat = torch.cat([p.grad.reshape(-1).double() for p in params])
            dist.all_reduce(flat, group=group)
        return res, y_d.grad, nz_d.grad

    def timed(fn, steps):
        if group is not None:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        if group is not None:
            dist.barrier()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        if group is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()) / steps

    last = []                                                    # outputs of the latest step, for --dump-outputs

    def dev_step():
        last.clear()                                             # released before the next step allocates its own
        last.append(step(aux, y.detach(), noise.detach()))
    from svgp_vae_b200 import step as step_mod
    prof, coll = None, {}
    for w in range(args.warmup):
        if args.lean and w == args.warmup - 1:
            be.start_profile()
            if world > 1:
                step_mod.start_coll_profile()
        dev_step()
        if args.lean and w == args.warmup - 1:
            prof = be.stop_profile()
            coll = step_mod.stop_coll_profile() if world > 1 else {}
    l0 = be.launches
    with ClockSampler(local) as clocks:
        ms = timed(dev_step, args.steps)
    launches = (be.launches - l0) // max(args.steps, 1)
    if args.dump_outputs and rank == 0:
        res, gy, gn = last[0]
        arrays = {k: v for k, v in res.items() if isinstance(v, torch.Tensor)}
        arrays.update(grad_y=gy, grad_noise=gn)
        arrays.update(("grad_" + k, p.grad) for k, p in svgp.named_parameters() if p.grad is not None)
        dump_outputs(args.dump_outputs, arrays, N)
    last.clear()

    # per-kernel device times of one more step (CUDA events on the launch stream)
    if prof is None:
        be.start_profile()
        if world > 1:
            step_mod.start_coll_profile()
        dev_step()
        prof = be.stop_profile()
        coll = step_mod.stop_coll_profile() if world > 1 else {}
        last.clear()

    # e2e: pinned host buffers in, results out, every step
    if args.lean:
        ms_e2e, h2d, d2h = float("nan"), 0, 0
    h_aux, h_y, h_nz = ((t.detach().cpu().pin_memory() for t in (aux, y, noise)) if not args.lean else (None, None, None))
    h_out = [torch.empty((N, L), dtype=torch.float32).pin_memory() for _ in range(4)] if not args.lean else []

    def e2e_step():
        a = h_aux.to(dev, non_blocking=True); yy = h_y.to(dev, non_blocking=True); nn = h_nz.to(dev, non_blocking=True)
        res, gy, gn = step(a, yy, nn)
        for dst, src in zip(h_out, (res["p_m"], res["p_v"], gy, gn)):
            dst.copy_(src.detach(), non_blocking=True)
        float(res["KL_term"])                                     # scalar read-back (syncs)
    if not args.lean:
        e2e_step()
        ms_e2e = timed(e2e_step, max(1, min(args.steps, 3)))
        h2d = sum(t.numel() * t.element_size() for t in (h_aux, h_y, h_nz))
        d2h = sum(t.numel() * t.element_size() for t in h_out) + 8

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:  # noqa: BLE001
            pass
        f16_run = measure_f16_peak(dev)
        peak = peaks.get("bf16_tflops_sustained")
        peak_src = "MEASURED_PEAKS.json bf16_tflops_sustained (kernel timed inside a long step)"
        if not peak:
            peak, peak_src = 1400.0, "fallback of B200_PROFILING.md (sustained ~1.4 PFLOP/s): MEASURED_PEAKS.json absent"
        f_alg = 9.0 * L * M * M * N                     # per GPU per step (SURVEY 8d)
        t_s = ms * 1e-3
        # dominant kernel of the step = the entry point with the largest total device time; its launch = the longest call
        top = max(prof.items(), key=lambda kv: kv[1]["ms"]) if prof else ("", {"ms": float("nan"), "calls": 0, "max_ms": float("nan")})
        top_name, top_ms = top[0], top[1]["max_ms"]
        # algorithmic FLOPs of one launch (2 x MACs) and the MMAs issued per algorithmic MAC in bf16-equivalents: the integer
        # path issues 10 kind::i8 MMAs (digit-plane pairs) per MAC at twice the kind::f16 rate (profiles/r02_i8_mma_probe.jsonl)
        # = 5 bf16-equivalents; the fp16 path issues 3.  scaled_gemm = 2L full N x M x M products; syrk = lower triangle of
        # L products; rowquad (triangular factor) = half of L full products
        # (three-leading-digit products, step.py: the adjoint SYRK and the S - Kinv half of pass D issue 8 instead of 10 pairs
        # up to M = 2048 -> e = 4 for them, 4.5 for the pass-D launch as a whole)
        d3 = be.use_i8 and M <= 2048 and os.environ.get("SVGP_I8_D3", "1") != "0"
        kern_alg = {"svgp_scaled_gemm_i8": (2.0 * N * M * M * (2 * L), 4.5 if d3 else 5.0), "svgp_scaled_gemm": (2.0 * N * M * M * (2 * L), 3.0),
                    "svgp_syrk": (1.0 * N * M * M * L, (13.0 if M > 2048 else 5.0) if be.use_i8 else 3.0), "svgp_rowquad": (1.0 * N * M * M * L, 3.0)}
        top_flops, top_e = kern_alg.get(top_name, (float("nan"), float("nan")))
        # DRAM bytes of one launch of that kernel from the committed ncu capture of this exact workload (else null)
        traffic = None
        try:
            tr = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
            if (N, M, L) == (N_PER_GPU, M_IND, L_CH):
                traffic = tr.get(top_name)
        except Exception:  # noqa: BLE001
            pass
        achieved = top_e * top_flops / (top_ms * 1e-3) / 1e12
        # what the tensor kernels of this implementation really issue per step, in bf16-equivalent FLOPs: 2 SYRKs (N M^2 L each,
        # x5) + 1 triangular row quad (N M^2 L, x3) + the 2L-matrix product of pass D (2 N M^2 2L, x5)
        # above M = 2048 both SYRKs compute both triangles (x 2) and the forward one multiplies thirteen pairs (6.5)
        syrk_e = (2 * 6.5 + 2 * 5.0) if M > 2048 else (5.0 + (4.0 if d3 else 5.0))
        launched = (syrk_e + 3.0 + 4 * (4.5 if d3 else 5.0)) * L * N * M * M if be.use_i8 else 3 * (3.0 * L + 2.0 * (2 * L)) * N * M * M
        # K1 (the kernel-matrix builder) is the HBM-bound kernel of the path: fp16 hi/lo row planes + 4 + 4 int8 digit planes
        k1_name = "svgp_kernel_fwd_i8" if "svgp_kernel_fwd_i8" in prof else "svgp_kernel_fwd"
        k1_ms = prof.get(k1_name, {}).get("max_ms")
        k1_bytes = (12.0 if k1_name.endswith("i8") else 8.0) * N * M + N * 8 * 4
        hbm_peak = peaks.get("hbm_gbs")
        k1 = None
        if k1_ms:
            k1_gbs = k1_bytes / (k1_ms * 1e-3) / 1e9
            k1 = {"bound": "hbm", "kernel": k1_name + " (operand-plane builder: maxima pass + write pass, float64 kernel evaluation)",
                  "achieved": k1_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": k1_gbs / hbm_peak if hbm_peak else None, "kernel_ms": k1_ms,
                  "algorithmic_bytes": k1_bytes}
        line = {
            "metric": METRIC, "value": n_total / t_s, "unit": "datapoints/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms, "higher_is_better": True, "scaling": "strong" if args.strong else "weak", "vs_baseline": None,
            "dtype": "int8 digit planes on tcgen05 kind::i8 with exact int32 TMEM accumulation (SYRK, scaled GEMM: fp32-accurate operands, "
                     "no accumulation rounding) + 3 x FP16 split (row quads) + f64 MxM stage", "data": "synthetic",
            "config": workload_config(args, world),
            "impl_notes": {"operands": "K_nm operand planes: fp16 hi/lo + 2 x 4 int8 digit planes = %.1f GB per GPU" % (12.0 * N * M / 1e9),
                           "parallelism": "N-sharded x%d, all-reduce of A_l/v_l and their adjoints, channel-sharded f64 MxM stage" % world},
            "roofline": {"bound": "tensor", "kernel": top_name, "achieved": achieved, "peak": peak, "unit": "TFLOP/s (bf16-equivalent)",
                         "frac": achieved / peak if peak else None, "traffic": traffic,
                         "note": "achieved = e x algorithmic FLOPs of the kernel's launch / its CUDA-event duration inside the step; e = MMAs issued "
                                 "per algorithmic MAC in bf16-equivalents: 10 kind::i8 digit-plane MMAs at twice the bf16 rate = 5 (integer path; 8 pairs = 4 for the matrices multiplied with three leading digits), "
                                 "3 (fp16 split path); peak = %s; fp16 cuBLAS 8192^3 timed in this run: %.1f TFLOP/s" % (peak_src, f16_run),
                         "kernel_ms": top_ms, "kernel_algorithmic_tflops": top_flops / (top_ms * 1e-3) / 1e12, "e": top_e,
                         "step_algorithmic_tflops": f_alg / t_s / 1e12,
                         "step_tensor_flops_launched": launched, "step_tensor_tflops_launched": launched / t_s / 1e12,
                         "step_frac_of_peak": launched / t_s / 1e12 / peak if peak else None,
                         "f16_cublas_tflops_in_run": f16_run},
            "roofline_k1": k1,
            "kernels_ms": {k: round(v["ms"], 3) for k, v in sorted(prof.items(), key=lambda kv: -kv[1]["ms"])},
            "kernels_calls": {k: v["calls"] for k, v in prof.items()},
            "e2e": ({"value": n_total / (ms_e2e * 1e-3), "unit": "datapoints/s", "ms_per_step": ms_e2e, "h2d_bytes_per_step": h2d,
                     "d2h_bytes_per_step": d2h} if not args.lean else None),
            "gpu_launches": int(launches), "clocks": clocks.summary(),
        }
        line["max_mem_gb"] = round(torch.cuda.max_memory_allocated(dev) / 1e9, 2)
        line["k3_ms"] = round(sum(v["ms"] for k, v in prof.items() if k in ("svgp_gemm_f64", "svgp_trinv_f64", "svgp_chol_f64", "svgp_ltl_f64")), 3)
        if world > 1:
            line["collectives"] = {k: {"ms": round(v["ms"], 3), "calls": v["calls"], "bytes": v["bytes"]} for k, v in coll.items()}
        if not args.no_cpu_baseline and world == 1:           # CPU leg: rank 0 of the single-GPU run only
            line["cpu_baseline"] = cpu_baseline(args, n_total)
        print(json.dumps(line), flush=True)
    if group is not None:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
