"""Worker of tests/test_gpu_dp_sync_bn.py (one process per GPU, launched with torch.distributed.run): synchronised
BatchNorm (LcnEngine.dp_sync_batch_norm) on `world` GPUs, checked against one GPU on the concatenated batch --
  (1) the BN mean / rstd taps of every layer are bit-identical across ranks and equal the single-GPU engine's on the
      concatenated batch; so do the forward outputs;
  (2) eager forward + backward with the streamed exchange: the mean loss and the exchanged bucket (true gradients) equal
      the single-GPU ones (equal shards) or the float64 restatement of (1/W) sum_r L_r (tests/sharded_oracle.py, unequal
      shards); on the fp32 path at dropout 0.25 also the float64 oracle on the concatenated batch;
  (3) K graph-replayed dp_train_step(sync_bn=True) steps in modes p2p and packed keep the replicas bit-identical and
      follow the single-GPU trajectory on the concatenated batch;
  (4) an engine that turns sync off again computes what an engine that never turned it on computes (up to the
      run-to-run spread of the atomics in the BatchNorm reductions).
argv: path (bf16 | fp32), rows of rank 0, rows of the other ranks.  LCN_DP_SHARE_GPU=1: every rank on device 0 (one-GPU
machines: the exchange then goes through CUDA IPC within one device, the rendezvous through gloo).  Prints one JSON line
per rank; exit code 0 = every check held (every error is printed first)."""
import json
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from lcn_pose_b200 import dist as lcn_dist  # noqa: E402
from oracle import lcn_oracle as O  # noqa: E402
from lcn_pose_b200.engine import LcnEngine  # noqa: E402
from tests.gpu_helpers import rel_err, synth_xy  # noqa: E402
from tests.sharded_oracle import loss_and_grads_sharded  # noqa: E402

# device (sync, W GPUs) against device (one GPU, concatenated batch): same per-row arithmetic, statistics and gradient
# sums reduced in another order.  Device against the float64 oracle: the tolerances of tests/test_gpu_parity.py.
TOL = {"bf16": dict(stat=1e-4, out=1e-2, grad=1e-2, oracle=1e-1), "fp32": dict(stat=1e-5, out=1e-4, grad=1e-4, oracle=2e-3)}


def main():
    path, n0, n1 = sys.argv[1], int(sys.argv[2]), int(sys.argv[3])
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
    tol = TOL[path]
    sizes = [n0] + [n1] * (world - 1)
    equal = len(set(sizes)) == 1
    steps, L = 4, 2
    errs, fails = {}, []

    def check(name, val, bound):
        errs[name] = val
        if not val < bound:
            fails.append(f"{name}={val:.3g} >= {bound:.3g}")

    nm = O.get_neighbour_matrix_by_hand(knn=3)
    cfg = O.LcnConfig(F=64, num_layers=L, neighbour_matrix=nm, regularization=0.0)

    def engine(sync):
        eng = LcnEngine(F=64, in_F=2, num_layers=L, neighbour_matrix=nm, path=path, device=f"cuda:{local}")
        eng.init_params(seed=42)
        lcn_dist.broadcast_parameters(eng.params)
        if sync is not None:
            lcn_dist.init_native_dp(eng, sync_bn=sync)
        return eng

    # every rank its own shard of one global batch (rank-seeded, so the shards differ)
    xs, ys = zip(*[synth_xy(n, seed=300 + r) for r, n in enumerate(sizes)])
    x_cat, y_cat = np.concatenate(xs), np.concatenate(ys)
    r0 = sum(sizes[:rank])
    xd = torch.as_tensor(xs[rank]).to(dev)
    yd = torch.as_tensor(ys[rank]).to(dev)
    n = sizes[rank]

    eng = engine(True)
    ref = engine(None)                          # one GPU, the concatenated batch, never connected
    p64 = {k: v.astype(np.float64) for k, v in eng.get_params().items()}
    xcd, ycd = torch.as_tensor(x_cat).to(dev), torch.as_tensor(y_cat).to(dev)
    n_bn = 1 + 2 * L

    # ---- (1) statistics and outputs of the forward pass ----
    out = eng.forward(xd, bn_group=n, training=True).cpu().numpy()
    taps = torch.stack([torch.stack([eng.read_tensor(k, l, n, n)[0] for k in (4, 5)]) for l in range(n_bn)])
    out_ref = ref.forward(xcd, bn_group=x_cat.shape[0], training=True).cpu().numpy()
    taps_ref = torch.stack([torch.stack([ref.read_tensor(k, l, x_cat.shape[0], x_cat.shape[0])[0] for k in (4, 5)])
                            for l in range(n_bn)])
    t0 = taps.clone()
    dist.broadcast(t0, src=0)
    taps_identical = bool(torch.equal(t0, taps))
    if not taps_identical:
        fails.append("BN statistics differ across ranks")
    check("bn_mean", rel_err(taps[:, 0].cpu().numpy(), taps_ref[:, 0].cpu().numpy()), tol["stat"])
    check("bn_rstd", rel_err(taps[:, 1].cpu().numpy(), taps_ref[:, 1].cpu().numpy()), tol["stat"])
    check("forward_out", rel_err(out, out_ref[r0:r0 + n]), tol["out"])

    # ---- (2) eager forward + backward, streamed exchange inside backward ----
    loss = eng.backward(xd, yd).clone()
    dist.all_reduce(loss)
    g = eng.unflatten(eng.true_grads())
    if equal:
        loss_ref = float(ref.backward(xcd, ycd).item())
        g_ref = ref.unflatten(ref.true_grads())
    else:
        loss_ref, g_ref, _ = loss_and_grads_sharded(cfg, p64, list(xs), list(ys))
    check("loss", abs(float(loss.item()) / world - loss_ref) / loss_ref, tol["out"])
    biases = O.bias_names(cfg)[:-1]               # in front of BatchNorm: the true gradient is 0, values are rounding
    scale = max(np.abs(v).max() for v in g_ref.values())
    gb = 0.0
    for k in g_ref:
        if k in biases:
            gb = max(gb, float(np.abs(g[k] - g_ref[k]).max() / scale))
        else:
            check(f"grad {k}", rel_err(g[k], g_ref[k]), tol["grad"] if equal else tol["oracle"])
    check("grad pre-BN biases (to max |grad|)", gb, tol["grad"] if equal else tol["oracle"])
    if path == "fp32":
        # dropout 0.25: the keep masks of every rank's rows, concatenated, into the float64 oracle
        rate = 0.25
        eng.forward(xd, bn_group=n, training=True, dropout=rate)
        loss = eng.backward(xd, yd, rate).clone()
        dist.all_reduce(loss)
        g = eng.unflatten(eng.true_grads())
        keep = [eng.dropout_keep(l, n, rate).cpu().numpy().astype(bool) for l in range(n_bn)]
        parts = [None] * world
        dist.all_gather_object(parts, keep)
        keep_shards = parts
        if equal:
            keep_cat = [np.concatenate([k[l] for k in parts]) for l in range(n_bn)]
            loss_o, g_o = O.loss_and_grads(cfg, p64, x_cat.astype(np.float64), y_cat.astype(np.float64), rate, keep_cat)
        else:
            loss_o, g_o, _ = loss_and_grads_sharded(cfg, p64, list(xs), list(ys), keep_shards, rate)
        check("dropout loss vs oracle", abs(float(loss.item()) / world - loss_o) / loss_o, 1e-4)
        worst = max(rel_err(g[k], g_o[k]) for k in g_o if k not in biases)
        check("dropout grads vs oracle", worst, tol["oracle"])

    # ---- (3) graph-replayed steps: replicas bit-identical, single-GPU trajectory ----
    traj = {}
    if equal:
        single = engine(None)
        s_losses = []
        for _ in range(steps):
            lo, _ = single.train_step_graph(xcd, ycd)
            s_losses.append(float(lo.item()))
    for mode in ("p2p", "packed"):
        e2 = engine(None)
        losses = []
        for _ in range(steps):
            lo, _ = lcn_dist.dp_train_step(e2, xd, yd, mode=mode, sync_bn=True)
            lt = lo.clone()
            dist.all_reduce(lt)
            losses.append(float(lt.item()) / world)
        flat = torch.cat([e2.params, e2.adam_m, e2.adam_v])
        r = flat.clone()
        dist.broadcast(r, src=0)
        if not torch.equal(flat, r):
            fails.append(f"{mode}: replicas diverged")
        traj[mode] = {"losses": losses}
        if equal:
            d = (e2.params - single.params).abs()
            keep_p = torch.ones_like(d, dtype=torch.bool)
            for b in biases:                       # Adam steps driven by rounding noise on both sides
                off, rows, cols = e2.tensors[b]
                keep_p[off:off + rows * cols] = False
            out_frac = float(((d > 1e-6 + 1e-4 * single.params.abs()) & keep_p).float().mean())
            check(f"{mode}: params off the single-GPU trajectory (fraction)", out_frac, 1e-3)
            check(f"{mode}: loss trajectory", max(abs(a - b) / b for a, b in zip(losses, s_losses)), tol["out"])
            traj[mode]["single_losses"] = s_losses
        e2.close()

    # ---- (4) sync off again == never on ----
    e_off = engine(True)
    e_off.dp_sync_batch_norm(False)
    e_never = engine(False)
    res = []
    for e in (e_off, e_never, e_never):
        o = e.forward(xd, bn_group=n, training=True).clone()
        e.backward(xd, yd)
        res.append(torch.cat([o.flatten(), e.grads_raw.clone()]))
    # the BatchNorm sums are reduced with atomics, so one engine is not bit-reproducible from run to run: the bound is
    # that run-to-run spread, floored at the statistics tolerance
    d_off = rel_err(res[0].cpu().numpy(), res[1].cpu().numpy())
    d_rr = rel_err(res[2].cpu().numpy(), res[1].cpu().numpy())
    errs["off_vs_never"], errs["never_run_to_run"] = d_off, d_rr
    if d_off > max(4 * d_rr, tol["stat"]):
        fails.append(f"sync off differs from never on: {d_off:.3g} (run to run {d_rr:.3g})")

    print(json.dumps({"rank": rank, "world": world, "path": path, "sizes": sizes, "taps_identical": taps_identical,
                      "errors": errs, "trajectories": traj, "fails": fails}), flush=True)
    for e in (eng, ref, e_off, e_never):
        e.close()
    dist.barrier()
    dist.destroy_process_group()
    sys.exit(1 if fails else 0)


if __name__ == "__main__":
    main()
