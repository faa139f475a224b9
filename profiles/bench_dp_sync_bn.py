"""Cost of synchronised BatchNorm (LcnEngine.dp_sync_batch_norm) in a data-parallel train step: graph-replayed
dp_train_step in mode p2p with sync off and on, alternated in rounds on the same engines, at the bench.py config (L=3,
F=64, knn=3, bf16, dropout 0.25) and two per-GPU batches: 4096 (bench.py) and the reference's batch_size 200 split over
the ranks.  Prints one JSON line (rank 0) with ms/step and poses/s (global) for both, the step count, and the GPU name and
power limit read in the same run.
    python -m torch.distributed.run --nproc-per-node N --master-addr 127.0.0.1 profiles/bench_dp_sync_bn.py [steps] [rounds]"""
import json
import os
import subprocess
import sys
import time

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402
from lcn_pose_b200 import dist as lcn_dist  # noqa: E402


def gpu_info(local):
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(local)],
                       capture_output=True, text=True, timeout=60)
    return q.stdout.strip()


def main():
    steps = int(sys.argv[1]) if len(sys.argv) > 1 else 200
    rounds = int(sys.argv[2]) if len(sys.argv) > 2 else 5
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    rows = {"per_gpu_4096": 4096, "reference_200": 200 // world}
    result = {"world": world, "steps_per_round": steps, "rounds": rounds, "gpu": gpu_info(local), "mode": "p2p"}
    for name, n in rows.items():
        x, y = bench.synth_xy(n, seed=1234 + rank)
        xd, yd = torch.as_tensor(x).to(dev), torch.as_tensor(y).to(dev)
        engs = {s: bench.make_engine(2, "bf16", local) for s in (False, True)}
        for s, e in engs.items():                  # capture + warm-up
            for _ in range(10):
                lcn_dist.dp_train_step(e, xd, yd, 0.25, mode="p2p", sync_bn=s)
        torch.cuda.synchronize()
        ms = {False: [], True: []}
        for _ in range(rounds):
            for s, e in engs.items():
                dist.barrier()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for _ in range(steps):
                    lcn_dist.dp_train_step(e, xd, yd, 0.25, mode="p2p", sync_bn=s)
                torch.cuda.synchronize()
                ms[s].append((time.perf_counter() - t0) / steps * 1e3)
        t = torch.tensor([min(ms[False]), min(ms[True])], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)   # a step ends when the slowest rank ends
        off, on = float(t[0]), float(t[1])
        result[name] = {"rows_per_gpu": n, "ms_per_step_sync_off": off, "ms_per_step_sync_on": on,
                        "poses_per_s_sync_off": n * world / off * 1e3, "poses_per_s_sync_on": n * world / on * 1e3,
                        "sync_cost_us_per_step": (on - off) * 1e3,
                        "ms_all_rounds": {"off": ms[False], "on": ms[True]}}
        for e in engs.values():
            e.close()
    if rank == 0:
        print(json.dumps(result), flush=True)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
