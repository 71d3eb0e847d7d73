"""The sharded step (torch.distributed group) on the CUDA kernels against the float64 oracle evaluated on the GPU.

tests/test_dist_gloo.py runs the multi-rank host logic on the float64 CPU stand-in, whose K_nm is never in a tensor-core
format; the branches that exist only for those formats run here: the all-gather of the int8 digit planes and their scales
(or of the fp16 hi/lo planes) in the chunked, channel-sharded backward, and the per-shard digit grids (column scales, the
SYRK's weight grid, the pair-bias terms) whose products are then summed over the ranks.  Every case spawns its ranks once
(tests/probes/parity_sharded.py): NCCL with one GPU per rank when there are enough devices, gloo on cuda:0 otherwise.

Each case checks the ten quantities of the sharded run AND of a single-process control on the whole batch to 1e-4 of
max|oracle|, and that the global outputs are bit-identical on every rank."""
import json
import os
import sys

import pytest

pytestmark = pytest.mark.gpu
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "probes"))

# the K_nm format every rank must have run on: "i8" integer tensor cores, "fp16" hi/lo tensor cores, "simt" fp32 SIMT
CASES = {
    # replicated K3 (L % W != 0); A_l / dS_l all-reduced from per-shard digit grids
    "A-replicated": (dict(N=65536, M=1024, L=3, world=2), "i8"),
    # channel-sharded K3 in one chunk, ragged shards
    "B-sharded-ragged": (dict(N=65536, M=1024, L=4, world=2, shard_rows=(30001, 35535)), "i8"),
    # channel-sharded chunked stage: int8 plane + scale all-gather, per-chunk factor gather into q1 column slices
    "C-sharded-chunked": (dict(N=65536, M=1024, L=4, world=2, mm_chunk=1), "i8"),
    # replicated chunked stage
    "D-replicated-chunked": (dict(N=65536, M=1024, L=3, world=2, mm_chunk=1), "i8"),
    # odd world: q1 column offsets r * L_own + off up to r = 2
    "E-three-ranks": (dict(N=49152, M=1024, L=6, world=3, shard_rows=(16000, 16384, 16768), mm_chunk=1), "i8"),
    # configs[4]'s M on 8 GPUs: one chunk of channels per rank, thirteen-pair full SYRK, debiased scaled GEMM
    "F-M4096-sharded": (dict(N=16384, M=4096, L=2, world=2), "i8"),
    # configs[4]'s M on 2 or 4 GPUs: the chunked channel-sharded stage
    "G-M4096-sharded-chunked": (dict(N=16384, M=4096, L=4, world=2, mm_chunk=1), "i8"),
    # fp16 engine (SVGP_TC_I8=0): hi/lo/inv all-gather
    "H-fp16-sharded-chunked": (dict(N=16384, M=256, L=4, world=2, mm_chunk=1, i8=False), "fp16"),
    # one shard below the tensor-core size (tc_min_rows = 2048): the whole group runs on the SIMT kernels
    "I-straddling": (dict(N=5632, M=256, L=4, world=2, shard_rows=(4096, 1536)), "simt"),
    "I-straddling-chunked": (dict(N=5632, M=256, L=4, world=2, shard_rows=(4096, 1536), mm_chunk=1), "simt"),
}
QUANTITIES = ("p_m", "p_v", "recon_l", "kl_l", "ce_l", "KL_term", "dy", "dnoise", "dhyp", "dZ")


@pytest.mark.parametrize("case", list(CASES))
def test_sharded_step_against_float64_oracle(cuda_backend, case):
    import parity_sharded
    kw, engine = CASES[case]
    o = parity_sharded.run(**kw)
    print(json.dumps(dict(case=case, **o)))
    for run in ("sharded", "control"):
        for k in QUANTITIES:
            assert o[run][k] < 1e-4, (run, k, o)
    # recon_l, kl_l, ce_l, KL_term, mu_hat and A_hat: gathered or replicated, the same bits on every rank
    assert all(o["same_across_ranks"].values()), o
    assert o["engine"] == [engine] * kw["world"], o
