"""Parity of the sharded step (torch.distributed group, CUDA kernels) against the float64 oracle evaluated on the GPU.

The whole batch of configs.sweep_inputs is built once; rank r gets rows [sum(shards[:r]), sum(shards[:r + 1])).  Each rank
takes J_r = <gm_r, p_m_r> + <gv_r, p_v_r> + KL_term / W (the gradient convention of INTEGRATION.md), so the ranks' J sum to
the J of parity_fullsize, whose streamlined float64 oracle on the whole batch is the reference.  A single-process step on the
whole batch (tc=True) is the control: when it passes and the sharded run does not, the multi-rank path is at fault.

NCCL with one GPU per rank when there are enough devices, otherwise gloo with every rank on cuda:0.
Usage: python tests/probes/parity_sharded.py N M L WORLD [mm_chunk] [shard rows ...] -> one JSON line."""
import json
import os
import socket
import subprocess
import sys
import tempfile
from datetime import timedelta

import torch
import torch.distributed as dist
import torch.multiprocessing as mp

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from parity_fullsize import objective, oracle, upstream  # noqa: E402  (also puts the repository and tests/ on sys.path)
import svgp_vae_b200 as pkg  # noqa: E402
from svgp_vae_b200 import backend, configs  # noqa: E402

QUANTITIES = ("p_m", "p_v", "recon_l", "kl_l", "ce_l", "KL_term", "dy", "dnoise", "dhyp", "dZ")
GLOBAL = ("recon_l", "kl_l", "ce_l", "KL_term", "mu_hat", "A_hat")      # identical on every rank


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).abs().max() / b.abs().max())


def _step(s, aux, y, noise, gm, gv, world=1, **kw):
    """elbo_step and the gradients of objective() -> dict of the ten quantities (CPU) and the raw result."""
    yy, nn = y.clone().requires_grad_(True), noise.clone().requires_grad_(True)
    res = s.elbo_step(aux, yy, nn, **kw)
    dy, dn, dZ, dh = torch.autograd.grad(objective(res, gm, gv, world), [yy, nn, s.inducing_index_points, s._hyp()])
    out = {k: res[k].detach().cpu() for k in ("p_m", "p_v", "recon_l", "kl_l", "ce_l")}
    out.update(KL_term=float(res["KL_term"].detach()), dy=dy.cpu(), dnoise=dn.cpu(), dZ=dZ.double(), dhyp=dh.double())
    return out, res


def _engine(calls):
    """Which K_nm format a rank's step ran on, from the entry points it called."""
    if "svgp_kernel_fwd_i8" in calls:
        return "i8"
    return "fp16" if "svgp_gemm_nn_tc" in calls else "simt"


def _worker(rank, world, port, tmp, ctor, mm_chunk, i8, nccl):
    os.environ["SVGP_TC_I8"] = "1" if i8 else "0"          # read when the backend is created, below
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dev = torch.device("cuda", rank if nccl else 0)
    torch.cuda.set_device(dev)
    if nccl:
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev, timeout=timedelta(minutes=5))
    else:
        dist.init_process_group("gloo", rank=rank, world_size=world, timeout=timedelta(minutes=5))
    try:
        be = backend.get_backend()
        d = {k: v.to(dev) for k, v in torch.load(os.path.join(tmp, "in%d.pt" % rank)).items()}
        s = pkg.productSVGP(**ctor).to(dev)
        be.start_profile()
        out, res = _step(s, d["aux"], d["y"], d["noise"], d["gm"], d["gv"], world, group=dist.group.WORLD, mm_chunk=mm_chunk)
        out["engine"] = _engine(be.stop_profile())
        for k in ("dZ", "dhyp"):
            dist.all_reduce(out[k])
            out[k] = out[k].cpu()
        same = {}
        for k in GLOBAL:
            t = res[k].detach().reshape(-1).contiguous()
            t0 = t.clone()
            dist.broadcast(t0, src=0)
            same[k] = torch.equal(t0, t)
        out["same"] = same
        torch.save(out, os.path.join(tmp, "out%d.pt" % rank))
    finally:
        dist.destroy_process_group()


def _gpu():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.splitlines()
    return q[0].strip() if q else torch.cuda.get_device_name(0)


def run(N, M, L, world, shard_rows=None, mm_chunk=None, i8=True, seed=1234):
    dev = torch.device("cuda")
    if shard_rows is None:
        q, r = divmod(N, world)
        shard_rows = [q + (i < r) for i in range(world)]
    shards = [int(n) for n in shard_rows]
    assert len(shards) == world and sum(shards) == N, (shards, N, world)
    cfg = configs.sweep_inputs(N, M, L, device=dev, seed=seed)
    s = pkg.productSVGP(**cfg["ctor"]).to(dev)
    gm, gv = upstream(N, L, dev)
    ref = oracle(cfg, s.inducing_index_points, gm, gv)
    ref = {k: v.cpu() if torch.is_tensor(v) else v for k, v in ref.items()}
    torch.cuda.empty_cache()

    be = backend.get_backend()
    use_i8 = be.use_i8
    be.use_i8 = i8
    try:
        ctl, _ = _step(s, cfg["aux"], cfg["y"], cfg["noise"], gm, gv, tc=True, mm_chunk=mm_chunk)
    finally:
        be.use_i8 = use_i8
    torch.cuda.empty_cache()

    ndev = torch.cuda.device_count()
    nccl = ndev >= world
    with tempfile.TemporaryDirectory() as tmp:
        r0 = 0
        for r, n in enumerate(shards):
            sl = slice(r0, r0 + n)
            r0 += n
            torch.save({k: t[sl].cpu() for k, t in (("aux", cfg["aux"]), ("y", cfg["y"]), ("noise", cfg["noise"]), ("gm", gm), ("gv", gv))},
                       os.path.join(tmp, "in%d.pt" % r))
        ctor = cfg["ctor"]
        del cfg, gm, gv
        torch.cuda.empty_cache()
        mp.spawn(_worker, args=(world, _free_port(), tmp, ctor, mm_chunk, i8, nccl), nprocs=world, join=True)
        outs = [torch.load(os.path.join(tmp, "out%d.pt" % r)) for r in range(world)]

    sh = {k: torch.cat([o[k] for o in outs]) for k in ("p_m", "p_v", "dy", "dnoise")}
    sh.update({k: outs[0][k] for k in ("recon_l", "kl_l", "ce_l", "KL_term", "dZ", "dhyp")})

    def errs(x, y):
        return {k: (abs(x[k] - y[k]) / abs(y[k]) if k == "KL_term" else _rel(x[k], y[k])) for k in QUANTITIES}

    return dict(N=N, M=M, L=L, world=world, shards=shards, mm_chunk=mm_chunk, i8=i8, seed=seed,
                collective="nccl" if nccl else "gloo", devices=ndev, gpu=_gpu(),
                sharded=errs(sh, ref), control=errs(ctl, ref), sharded_vs_control=errs(sh, ctl),
                same_across_ranks={k: all(o["same"][k] for o in outs) for k in GLOBAL},
                engine=[o["engine"] for o in outs])


if __name__ == "__main__":
    a = [int(x) for x in sys.argv[1:]]
    o = run(*a[:4], mm_chunk=a[4] if len(a) > 4 and a[4] else None, shard_rows=a[5:] or None)
    print(json.dumps(o), flush=True)
