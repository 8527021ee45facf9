#!/usr/bin/env python
"""Slice-sampled hypers on row-sharded replicas (run with torchrun, one rank per GPU).

Every rank holds its row shard and a replica of the suffstats.  After row-sharded sweeps with the delta all-reduce inside
the C ABI (msb_state_allreduce_deltas), the replicas are bit-identical, so msb_state_slice_hp with the same
(seed, counter) must give every rank the same hypers and alpha, bit for bit, with no collective of their own.  Prints one
line per iteration and "all ok" / "FAILED"; exit status 0 / 1."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import common_b200 as cb  # noqa: E402
from common_b200 import hyperprior as hpr  # noqa: E402
from common_b200 import dist as cbd  # noqa: E402

N_PER_RANK, K, ITERS = 40000, 12, 3


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=device)
    ctx = cb.Context(local)
    torch.cuda.set_stream(torch.cuda.ExternalStream(ctx.stream(), device=device))
    comm = cbd.NcclComm(ctx, rank, world)
    descs = [cb.bb, cb.nich, cb.niw(3), cb.gp, cb.dd(9)]
    n = N_PER_RANK
    arr, z = cb.synth.make_dataset(descs, n, K, seed=5, stream=rank)
    st = cb.state(ctx, descs, max_groups=K + 4, cluster_hp={"alpha": 1.0})
    st.bind(cb.numpy_dataview(arr))
    gids = np.asarray([st.create_group() for _ in range(K + 2)])     # two groups stay empty
    cbd.add_values_sharded(st, gids[z], device, comm, n * world)
    e1 = hpr.log_exponential(1.0)
    hparams = {0: {("alpha", "beta"): (hpr.log_noninformative_beta_prior, 1.0)},
               1: {"mu": (hpr.log_normal(0.0, 10.0), 0.5), "kappa": (e1, 1.0), "sigmasq": (e1, 1.0), "nu": (e1, 2.0)},
               2: {"kappa": (e1, 1.0), "nu": (hpr.log_exponential(0.1), 3.0)}, 3: {"alpha": (e1, 1.0), "inv_beta": (e1, 0.5)}}
    ok = True
    for it in range(ITERS):
        st.sweep(seed=9, sweep=it, row_id_offset=rank * n, defer_apply=True, wait=False)
        st.allreduce_deltas(comm, n * world)
        r = st.slice_hp(hparams, {"alpha": (e1, 1.0)}, seed=21, counter=it)
        mine = {"groups": st.groups(), "capped": r["capped"],
                "values": {str(d): np.asarray(list(v.values()) if isinstance(v, dict) else [v]).tobytes() for d, v in r["values"].items()},
                "hp": [np.concatenate([np.ravel(v) for v in st.get_component_hp(d).values()]).tobytes() for d in range(len(descs))]}
        gathered = [None] * world
        dist.all_gather_object(gathered, mine)
        same = all(g == gathered[0] for g in gathered)
        ok &= same and r["capped"] == 0
        if rank == 0:
            print("iteration %d: %d ranks hold identical hypers (%d specs, alpha %.6g): %s (capped %d)"
                  % (it, world, sum(len(v) if isinstance(v, dict) else 1 for v in r["values"].values()), r["values"]["alpha"],
                     same, r["capped"]))
    if rank == 0:
        print("all ok" if ok else "FAILED")
    st.close()
    comm.close()
    dist.destroy_process_group()
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
