#!/usr/bin/env python
"""Hyperparameter draws on row-sharded replicas (run with torchrun, one rank per GPU).

Every rank holds its row shard and a replica of the suffstats.  After row-sharded sweeps with the delta all-reduce inside
the C ABI (msb_state_allreduce_deltas), the replicas are bit-identical, so msb_state_hp_gibbs with the same (seed,
counter) must give every rank the same weights, bit for bit, the same draws and the same hypers -- with no collective of
its own.  Prints one line per iteration and "all ok" / "FAILED"; exit status 0 / 1."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import common_b200 as cb  # noqa: E402
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
    descs = [cb.dd(9), cb.nich, cb.gp, cb.bb, cb.bnb, cb.bbnc, cb.niw(3)]
    n = N_PER_RANK
    arr, z = cb.synth.make_dataset(descs, n, K, seed=5, stream=rank)
    st = cb.state(ctx, descs, max_groups=K + 2, cluster_hp={"alpha": 1.0})
    st.bind(cb.numpy_dataview(arr))
    gids = np.asarray([st.create_group() for _ in range(K)])
    cbd.add_values_sharded(st, gids[z], device, comm, n * world)
    rng = np.random.default_rng(3)      # the same grids on every rank
    st.set_hp_grid(0, [{"alphas": rng.uniform(0.2, 3.0, 9)} for _ in range(16)])
    st.set_hp_grid(1, [{"mu": m, "kappa": k, "sigmasq": s, "nu": v} for m, k, s, v in rng.uniform(0.2, 3.0, (16, 4))])
    st.set_hp_grid(2, [{"alpha": a, "inv_beta": b} for a, b in rng.uniform(0.2, 3.0, (16, 2))])
    st.set_hp_grid(3, [{"alpha": a, "beta": b} for a, b in rng.uniform(0.2, 3.0, (16, 2))])
    st.set_hp_grid(4, [{"alpha": a, "beta": b, "r": 1.0} for a, b in rng.uniform(1.5, 3.0, (16, 2))])
    st.set_hp_grid(5, [{"alpha": a, "beta": b} for a, b in rng.uniform(0.2, 3.0, (16, 2))])
    st.set_hp_grid(6, [{"mu": np.zeros(3), "kappa": k, "psi": np.eye(3) * s, "nu": 3.0 + v} for k, s, v in rng.uniform(0.2, 3.0, (16, 3))])
    st.set_cluster_hp_grid(np.exp(np.linspace(-3, 3, 32)))
    ok = True
    for it in range(ITERS):
        st.sweep(seed=9, sweep=it, row_id_offset=rank * n, defer_apply=True, wait=False)
        st.allreduce_deltas(comm, n * world)
        r = st.hp_gibbs(seed=21, counter=it, weights=True)
        mine = {"choice": r["choice"], "logw": {k: v.tobytes() for k, v in r["logw"].items()},
                "hp": [{k: np.asarray(v).tobytes() for k, v in st.get_component_hp(d).items()} for d in range(len(descs))],
                "alpha": st.get_cluster_hp()["alpha"]}
        gathered = [None] * world
        dist.all_gather_object(gathered, mine)
        same = all(g == gathered[0] for g in gathered)
        ok &= same
        if rank == 0:
            print("iteration %d: %d ranks draw identical logw bits, choices and hypers: %s (choices %s)" % (it, world, same, r["choice"]))
    if rank == 0:
        print("all ok" if ok else "FAILED")
    st.close()
    comm.close()
    dist.destroy_process_group()
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
