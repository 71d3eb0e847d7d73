"""Under a group every rank builds K_nm in the same format: the tensor-core formats only when EVERY shard is tensor-core sized.

The chunked, channel-sharded backward all-gathers the adjoint operand planes in the K_nm format (int8 digit planes and
scales, fp16 hi/lo/inv, or float64), so ranks that chose different formats would issue different collectives.  Two gloo
ranks on the float64 stand-in backend, whose `want_tc` here follows the CUDA backend's row threshold and whose K1 records
the `tc` flag it receives.  (The stand-in's K_nm has one format whatever the flag, so the collectives match either way.)"""
import os
import socket

import pytest
import torch.distributed as dist
import torch.multiprocessing as mp

from svgp_vae_b200 import configs

N_TRAIN, M, L = 8192, 32, 4


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, shards, out):
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root); sys.path.insert(0, os.path.join(root, "tests"))
    from oracle_backend import OracleBackend
    import svgp_vae_b200 as pkg
    from svgp_vae_b200 import backend

    class RowThresholdBackend(OracleBackend):
        def __init__(self):
            super().__init__()
            self.tc_flags = []

        def want_tc(self, N, M):
            return N >= 2048

        def kernel_fwd(self, spec, Fx, Fz, hyp, tc=False):
            self.tc_flags.append(bool(tc))
            return super().kernel_fwd(spec, Fx, Fz, hyp, tc=tc)

    be = RowThresholdBackend()
    backend.set_backend_for_tests(be)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    cfg = configs.sweep_inputs(sum(shards), M, L, N_train=N_TRAIN)
    s = pkg.productSVGP(**cfg["ctor"])
    sl = slice(sum(shards[:rank]), sum(shards[:rank + 1]))
    y = cfg["y"][sl].clone().requires_grad_(True)
    res = s.elbo_step(cfg["aux"][sl], y, cfg["noise"][sl], group=dist.group.WORLD, mm_chunk=1)
    (res["p_v"].sum() + res["KL_term"] / world).backward()
    out[rank] = dict(tc=be.tc_flags, b_total=res["b_total"])
    dist.destroy_process_group()


@pytest.mark.parametrize("shards,tc", [((4096, 1536), False), ((2048, 3584), True)])
def test_all_ranks_agree_on_the_knm_format(shards, tc):
    """4096 + 1536 rows: one shard is below 2048 rows, so both ranks run on the SIMT format (rank 0 alone would take the
    tensor cores).  2048 + 3584: both shards qualify and keep the tensor-core format."""
    world = len(shards)
    out = mp.Manager().dict()
    mp.spawn(_worker, args=(world, _free_port(), shards, out), nprocs=world, join=True)
    for r in range(world):
        # K1 of the data rows only: K_mm and kappa are built by kernel_fwd_f64 / kernel_diag_fwd
        assert out[r]["tc"] == [tc], (r, out[r])
        assert out[r]["b_total"] == float(sum(shards))
