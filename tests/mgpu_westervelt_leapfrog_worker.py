"""Worker of tests/test_gpu_westervelt_leapfrog.py on N >= 2 real GPUs:

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 \
        --master-port 29613 tests/mgpu_westervelt_leapfrog_worker.py --out /tmp/wl.json

The Westervelt leapfrog solve of one global box partitioned over the GPUs (peer-memory halo with graph
replay and eager launches, the NCCL halo, block and blob partitions) against the same solve on rank 0
alone (``selfcheck.multi_gpu_parity``)."""

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    a = ap.parse_args()
    import torch
    import torch.distributed as dist

    rank = int(os.environ["RANK"])
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", rank)))
    dist.init_process_group("nccl", device_id=torch.device("cuda", torch.cuda.current_device()))
    from fenicsx_fus_gpu_b200.selfcheck import multi_gpu_parity

    base = dict(workload="westervelt", integrator="leapfrog", P=4, n_per_rank=5, nsteps=10)
    cases = [
        dict(dtype=np.float64),
        dict(dtype=np.float64, use_graph=False),
        dict(dtype=np.float64, halo_kind="nccl"),
        dict(dtype=np.float64, partition="blob"),
        dict(dtype=np.float32),
    ]
    results = [multi_gpu_parity(**base, **c) for c in cases]
    if rank == 0:
        for r in results:
            print(f"[mgpu] westervelt leapfrog {r['dtype']} {r['partition']} halo={r['halo']} graph={r['graph']}: "
                  f"rel-L2 u {r['rel_l2_u']:.2e} v {r['rel_l2_v']:.2e} {'ok' if r['ok'] else 'FAIL'}", flush=True)
        with open(a.out, "w") as f:
            json.dump(dict(ok=all(r["ok"] for r in results), parity=results), f)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
