"""Worker of tests/test_gpu_dp.py (one process per GPU, launched with torch.distributed.run): data-parallel LCN training
on `world` GPUs, checked on hardware --
  * the exchanged gradient bucket equals the mean of the ranks' local buckets (bit-wise up to the reduction order:
    compared against an fp64 mean of the all-gathered local buckets),
  * after K graph-replayed DP steps every replica holds bit-identical parameters and Adam moments,
  * the replicas' trajectory equals a single process that averages the same per-rank gradients itself.
argv: mode (p2p | p2p-end | packed).  LCN_DP_SHARE_GPU=1: every rank on device 0 (one-GPU machines: the exchange then
goes through CUDA IPC within one device, the rendezvous through gloo).  Prints one JSON line per rank; exit code 0 = all
assertions held."""
import json
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from lcn_pose_b200 import dist as lcn_dist  # noqa: E402
from lcn_pose_b200.engine import LcnEngine  # noqa: E402
from lcn_pose_b200.tools import params_help  # noqa: E402
from tests.gpu_helpers import synth_xy  # noqa: E402


def stage(msg):
    if os.environ.get("LCN_DP_TRACE"):
        print(f"[rank {os.environ.get('RANK')}] {msg}", file=sys.stderr, flush=True)


def main():
    if os.environ.get("LCN_HANG_TRACE"):          # debugging aid: dump every thread's Python stack after N seconds
        import faulthandler
        faulthandler.dump_traceback_later(float(os.environ["LCN_HANG_TRACE"]), exit=False)
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    shared = os.environ.get("LCN_DP_SHARE_GPU") == "1"
    if shared:
        local = 0
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if shared:
        dist.init_process_group("gloo")
    else:
        dist.init_process_group("nccl", device_id=dev)
    nm = params_help.get_neighbour_matrix_by_hand(params_help.filter_hub.neighbour_dict_set[0], knn=3)
    mode = sys.argv[1] if len(sys.argv) > 1 else "packed"
    steps, n = 5, 512

    def engine():
        e = LcnEngine(F=64, in_F=2, num_layers=1, neighbour_matrix=nm, path="bf16", device=f"cuda:{local}")
        e.init_params(seed=42)
        lcn_dist.broadcast_parameters(e.params)
        return e
    eng = engine()
    x, y = synth_xy(n, seed=100 + rank)                        # every rank its own shard of the global batch
    xd, yd = torch.as_tensor(x).to(dev), torch.as_tensor(y).to(dev)

    stage('engine built')
    # ---- (1) the exchanged bucket is the mean of the local buckets ----
    eng.forward(xd, bn_group=n, training=True, dropout=0.25)
    eng.backward(xd, yd, 0.25)
    local_bucket = eng.pack_grads().clone()
    gathered = [torch.empty_like(local_bucket) for _ in range(world)]
    dist.all_gather(gathered, local_bucket)
    mean64 = torch.stack([g.double() for g in gathered]).mean(0)
    lcn_dist.average_gradient_bucket(eng.grads_compact)
    err = float((eng.grads_compact.double() - mean64).abs().max() / mean64.abs().max())
    assert err < 1e-6, err
    eng.unpack_grads()
    eng.adam()
    stage('torch-level bucket mean ok')
    err_native = None
    if mode in ("p2p", "p2p-end"):
        # the exchange inside lcn_model_backward (streamed per layer behind the weight-gradient GEMMs, or one exchange at
        # the end) leaves the same mean in the bucket
        eng4 = engine()
        lcn_dist.init_native_dp(eng4)
        eng4.dp_enable(1 if mode == "p2p" else 2)
        stage('native communicator created')
        eng4.forward(xd, bn_group=n, training=True, dropout=0.25)
        eng4.backward(xd, yd, 0.25)
        torch.cuda.synchronize()
        stage('eager backward with the exchange inside finished')
        got = eng4.pack_grads().double()
        err_native = float((got - mean64).abs().max() / mean64.abs().max())
        assert err_native < 1e-5, err_native

    # ---- (2) K graph-replayed DP steps (what bench.py --gpus N runs): replicas stay bit-identical ----
    eng2 = engine()
    losses = []
    for i in range(steps):
        loss, _ = lcn_dist.dp_train_step(eng2, xd, yd, 0.25, mode=mode)
        losses.append(float(loss.item()))
        stage(f'graph step {i} done')
    flat = torch.cat([eng2.params, eng2.adam_m, eng2.adam_v])
    ref = flat.clone()
    dist.broadcast(ref, src=0)
    identical = bool(torch.equal(flat, ref))
    assert identical, "replicas diverged"
    assert eng2.step == steps

    # ---- (3) same trajectory as averaging the all-gathered per-rank gradients by hand (eager, no graph) ----
    eng3 = engine()
    for _ in range(steps):
        eng3.forward(xd, bn_group=n, training=True, dropout=0.25)
        eng3.backward(xd, yd, 0.25)
        b = eng3.pack_grads()
        parts = [torch.empty_like(b) for _ in range(world)]
        dist.all_gather(parts, b)
        b.copy_(torch.stack([q.double() for q in parts]).mean(0).float())
        eng3.unpack_grads()
        eng3.adam()
    d = (eng3.params - eng2.params).abs()
    outliers = int((d > 1e-6 + 1e-4 * eng2.params.abs()).sum())
    assert outliers <= 16 and float(d.max()) < 2e-4, (outliers, float(d.max()))
    print(json.dumps({"rank": rank, "world": world, "mode": mode, "bucket_mean_rel_err": err, "native_bucket_mean_rel_err": err_native, "replicas_identical": identical,
                      "losses": losses, "manual_avg_max_param_diff": float(d.max()), "outliers": outliers}), flush=True)
    for e in (eng, eng2, eng3) + ((eng4,) if err_native is not None else ()):
        e.close()
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
