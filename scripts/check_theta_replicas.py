#!/usr/bin/env python
"""bbnc parameter draws on row-sharded replicas (run with torchrun, one rank per GPU).

Every rank holds its row shard and a replica of the suffstats.  After row-sharded sweeps with the delta all-reduce inside
the C ABI (msb_state_allreduce_deltas), the replicas are bit-identical, so msb_state_redraw_empty followed by
msb_state_theta with the same (seed, counter) must give every rank the same p in every group, bit for bit, with no
collective of their own.  Prints one line per iteration and "all ok" / "FAILED"; exit status 0 / 1."""
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
    descs = [cb.bbnc, cb.dd(9), cb.bbnc, cb.nich, cb.bbnc]
    n = N_PER_RANK
    arr, z = cb.synth.make_dataset(descs, n, K, seed=5, stream=rank)
    st = cb.state(ctx, descs, max_groups=K + 4, cluster_hp={"alpha": 1.0})
    st.set_component_hp(2, {"alpha": 0.5, "beta": 2.0})
    st.bind(cb.numpy_dataview(arr))
    gids = np.asarray([st.create_group() for _ in range(K + 2)])     # two groups stay empty
    cbd.add_values_sharded(st, gids[z], device, comm, n * world)
    bbnc = [0, 2, 4]
    ok = True
    for it in range(ITERS):
        st.sweep(seed=9, sweep=it, row_id_offset=rank * n, defer_apply=True, wait=False)
        st.allreduce_deltas(comm, n * world)
        st.redraw_empty(seed=21, counter=it)
        capped = st.theta({0: {"p": 0.1}, 2: {"p": 1.0}, 4: {"p": 0.02}}, seed=21, counter=it)
        groups = st.groups()
        mine = {"groups": groups, "capped": capped,
                "p": [st.get_suffstats(d, g, "p").tobytes() for d in bbnc for g in groups],
                "empty": st.empty_groups()}
        gathered = [None] * world
        dist.all_gather_object(gathered, mine)
        same = all(g == gathered[0] for g in gathered)
        ok &= same and capped == 0
        if rank == 0:
            print("iteration %d: %d ranks hold identical p in %d groups x %d bbnc features: %s (capped %d, empty %s)"
                  % (it, world, len(groups), len(bbnc), same, capped, mine["empty"]))
    if rank == 0:
        print("all ok" if ok else "FAILED")
    st.close()
    comm.close()
    dist.destroy_process_group()
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
