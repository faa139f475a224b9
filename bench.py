#!/usr/bin/env python
"""bench.py -- poses/s of the LCN hot path on N B200s of one node (one process per GPU).

    python bench.py --gpus N --steps K --warmup W                    # this repo's CUDA path, BASELINE.json configs[1]
    python bench.py --impl reference --gpus N --steps K --warmup W   # the reference's CPU path (restated), same config
    python bench.py --config 3|4|5 ...                               # the other BASELINE.json configs (see CONFIGS)
    python bench.py ... --dump-outputs DIR                           # + what the last timed step computed, as DIR/<name>.npy

Prints ONE JSON line (rank 0).  `config` is identical in both arms (it names the workload, nothing else); how each arm
ran it is under `detail`.  See DESIGN.md "Measurement" for every field.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CONFIGS = {
    2: dict(knn=3, layers=3, F=64, mask="locally_connected", batch=4096,
            what="train step (fwd + bwd + masked TF1 Adam), BASELINE.json configs[1]"),
    3: dict(knn=3, layers=3, F=64, mask="locally_connected", batch=256,
            what="inference at BN group 256 -> denormalize -> Protocol-1 and Protocol-2 MPJPE, poses sharded by BN group, "
                 "BASELINE.json configs[2]"),
    4: dict(knn=3, layers=3, F=64, mask="exponential", batch=4096,
            what="train step on base + flip + rotate + translate augmented set (device gather per step), exponential mask, "
                 "data parallel, BASELINE.json configs[3]"),
    5: dict(knn=3, layers=5, F=128, mask="locally_connected", batch=16384,
            what="wide / deep sweep knn in {1,2,3,full}: train step + mid-layer GEMM vs mask density, BASELINE.json configs[4]"),
}


def nnz_of(mask, knn):
    return 289 if mask == "exponential" else {1: 57, 2: 111, 3: 175, 4: 237, 5: 273}.get(knn, 289)


def fwd_flop_per_pose(nnz, layers, F):
    return 2 * nnz * (2 * F + 2 * layers * F * F + 3 * F)            # SURVEY 8(d)


def workload_config(cfg_id, dropout):
    """The `config` object: identical in the GPU arm and the reference arm."""
    c = CONFIGS[cfg_id]
    return {"workload": f"LCN knn={c['knn']} layers={c['layers']} F={c['F']} {c['mask']} mask: {c['what']}",
            "config_id": cfg_id, "batch_per_gpu": c["batch"], "dropout": dropout,
            "l2": "GPU arm: L2 flushed between steps (256 MiB memset); CPU arm: not applicable"}


def synth_xy(n, seed=1234):
    rng = np.random.default_rng(seed)
    root = rng.uniform(-0.5, 0.5, (n, 1, 2))
    x = np.clip(root + rng.normal(0, 0.15, (n, 17, 2)), -1, 1)
    y = np.concatenate([x + rng.normal(0, 0.02, (n, 17, 2)), rng.normal(0, 0.1, (n, 17, 1))], axis=2)
    return x.reshape(n, 34).astype(np.float32), y.reshape(n, 51).astype(np.float32)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops", 1590.0), d.get("bf16_tflops_sustained", 1400.0), d.get("hbm_gbs", 6650.0), "measured"
    return 1590.0, 1400.0, 6650.0, "fallback"


def ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the committed
    `ncu --set full` capture (profiles/roofline_traffic.json names the report); None when absent."""
    p = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if not os.path.exists(p):
        return None
    d = json.load(open(p))
    return d.get("dram_bytes_read", 0) + d.get("dram_bytes_write", 0)


DUMP_BYTES = 60 << 20


def dump_outputs(out_dir, arrays):
    """Write each array as out_dir/<name>.npy, float32 kept and everything else as float64, at most DUMP_BYTES in all:
    when the arrays together are larger, each one over its share is replaced by a fixed, seeded sample of its elements
    (flattened), so that two runs with the same arguments write the same elements and can be compared one to one."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: np.asarray(v) for k, v in arrays.items()}
    arrays = {k: v if v.dtype == np.float32 else v.astype(np.float64) for k, v in arrays.items()}
    share = DUMP_BYTES // len(arrays)
    over = sum(a.nbytes for a in arrays.values()) > DUMP_BYTES
    for name, a in arrays.items():
        if over and a.nbytes > share:
            idx = np.sort(np.random.default_rng(0).choice(a.size, share // a.itemsize, replace=False))
            a = a.reshape(-1)[idx]
        np.save(os.path.join(out_dir, name + ".npy"), a)


class ClockSampler(threading.Thread):
    """SM clock + throttle reasons sampled during the timed region: NVML (about 1 ms per sample) when pynvml is
    importable, else nvidia-smi (about 100 ms per sample)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.rows = index, False, []

    def run(self):
        try:
            import pynvml as N
            N.nvmlInit()
            h = N.nvmlDeviceGetHandleByIndex(self.index)
            mx = N.nvmlDeviceGetMaxClockInfo(h, N.NVML_CLOCK_SM)
            pick = lambda new, old: getattr(N, new) if hasattr(N, new) else getattr(N, old)
            bits = [pick("nvmlClocksEventReasonHwSlowdown", "nvmlClocksThrottleReasonHwSlowdown"),
                    pick("nvmlClocksEventReasonHwThermalSlowdown", "nvmlClocksThrottleReasonHwThermalSlowdown"),
                    pick("nvmlClocksEventReasonSwThermalSlowdown", "nvmlClocksThrottleReasonSwThermalSlowdown"),
                    pick("nvmlClocksEventReasonSwPowerCap", "nvmlClocksThrottleReasonSwPowerCap")]
            get = getattr(N, "nvmlDeviceGetCurrentClocksEventReasons", None) or N.nvmlDeviceGetCurrentClocksThrottleReasons
            while not self.stop_flag:
                sm = N.nvmlDeviceGetClockInfo(h, N.NVML_CLOCK_SM)
                r = get(h)
                self.rows.append([str(sm), str(mx)] + ["Active" if (r & b) else "Not Active" for b in bits])
                time.sleep(0.002)
            return
        except Exception:
            pass
        self.run_smi()

    def run_smi(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i",
                                      str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        sm = sorted(int(r[0]) for r in self.rows if r[0].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None,
                "sm_max_mhz": int(self.rows[0][1]) if self.rows[0][1].isdigit() else None,
                "reasons": reasons, "samples": len(self.rows)}


# --------------------------------------------------------------------------------------------------
# CPU arm: the reference executes this path as dense fp32 matmuls on masked weights (TF stock ops,
# network/models_att.py).  TensorFlow is not installable here, so the restated graph
# (oracle/torch_restatement.py, autograd) + the oracle's TF1 Adam is timed on all host cores -- at the SAME batch,
# the SAME dropout rate (fresh uniform keep masks every step, as tf.nn.dropout draws them) and the SAME model.
# --------------------------------------------------------------------------------------------------
def cpu_train_steps(cfg_id, dropout, steps, warmup):
    import torch
    from oracle import lcn_oracle as O
    from oracle import torch_restatement as T
    c = CONFIGS[cfg_id]
    torch.set_num_threads(os.cpu_count() or 1)
    cfg = O.LcnConfig(F=c["F"], num_layers=c["layers"], mask_type=c["mask"],
                      neighbour_matrix=O.get_neighbour_matrix_by_hand(knn=c["knn"]))
    p = T.build_params(O.init_params(cfg, seed=42, dtype=np.float32), dtype=torch.float32)
    batch = c["batch"]
    x, y = synth_xy(batch)
    xt, yt = torch.tensor(x), torch.tensor(y)
    m = {k: torch.zeros_like(v) for k, v in p.items()}
    v2 = {k: torch.zeros_like(v) for k, v in p.items()}
    n_bn = 1 + 2 * c["layers"]
    t = 0

    def step():
        nonlocal t
        t += 1
        for v in p.values():
            v.grad = None
        keep = [(torch.rand((batch, 17 * c["F"])) >= dropout).float() for _ in range(n_bn)] if dropout > 0 else None
        loss, _ = T.loss_fn(cfg, p, xt, yt, dropout, keep)
        loss.backward()
        lr_t = O.learning_rate_at(cfg, t) * math.sqrt(1 - 0.999 ** t) / (1 - 0.9 ** t)
        with torch.no_grad():
            for k, w in p.items():
                if w.grad is None:
                    continue
                m[k].mul_(0.9).add_(w.grad, alpha=0.1)
                v2[k].mul_(0.999).addcmul_(w.grad, w.grad, value=0.001)
                w.sub_(lr_t * m[k] / (v2[k].sqrt() + 1e-8))
        return float(loss.detach())
    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = time.perf_counter() - t0
    return dt, torch.get_num_threads(), batch


def run_reference(args, rank, world):
    if rank != 0:
        return
    cfg_id = args.config if args.config in (2, 4) else 2
    dt, threads, batch = cpu_train_steps(cfg_id, args.dropout, args.steps, args.warmup)
    value = batch * args.steps / dt
    line = {"impl": "reference", "metric": "poses/sec (LCN train step)", "value": value, "unit": "poses/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(cfg_id, args.dropout),
            "detail": {"path": "dense fp32 matmuls on masked weights, torch-CPU autograd + TF1 Adam", "launch": "eager",
                       "parallelism": f"{threads} host threads, one process"},
            "cpu_baseline": {"value": value, "unit": "poses/s", "cores": threads, "kind": "port",
                             "sample": f"{args.steps} train steps at batch {batch}, dropout {args.dropout} (dense fp32 "
                                       f"restatement of the TF graph; TensorFlow 2.13 not installable offline)"},
            "e2e": {"value": value, "unit": "poses/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), file=JSON_OUT, flush=True)


# --------------------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------------------
def launches_per_step(n_bn, path, gather=False):
    """Kernels of this library per train step (counted from the launch list, profiles/r2): forward: (GEMM | first
    layer) + bn_act per BN layer (the BatchNorm statistics are accumulated by the GEMM itself on the bf16 path; the
    split-bf16 path adds k_bn_finalize), head; backward: loss, head dgrad, last-layer wgrad, BN backward (reduce + apply)
    per BN layer, dgrad + wgrad per mid layer, first-layer wgrad, bias-gradient reduce; optimizer: pairdot, mask gradient,
    Adam, 2 weight packs (mid layers; both edge layers)."""
    fwd = 2 * n_bn + 1 + (n_bn if path != "bf16" else 0)
    bwd = 3 + 2 * n_bn + 2 * (n_bn - 1) + 2
    opt = 5
    return fwd + bwd + opt + (1 if gather else 0)


def make_engine(cfg_id, path, local_rank, knn=None):
    from lcn_pose_b200.engine import LcnEngine
    from lcn_pose_b200.tools import filter_hub, params_help
    c = CONFIGS[cfg_id]
    knn = c["knn"] if knn is None else knn
    nm = params_help.get_neighbour_matrix_by_hand(filter_hub.neighbour_dict_set[0], knn=knn)
    eng = LcnEngine(F=c["F"], in_F=2, num_layers=c["layers"], mask_type=c["mask"], neighbour_matrix=nm, path=path,
                    device=f"cuda:{local_rank}")
    eng.init_params(seed=42)
    return eng


def run_gpu(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    try:
        if args.config == 3:
            line = run_config3(args, rank, world, local_rank, dev)
        elif args.config == 5:
            line = run_config5(args, rank, world, local_rank, dev)
        else:
            line = run_train(args, rank, world, local_rank, dev)
        if rank == 0 and line is not None:
            print(json.dumps(line), file=JSON_OUT, flush=True)
    finally:
        if world > 1:
            dist.destroy_process_group()


def barrier_fn(world):
    import torch
    import torch.distributed as dist

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()
    return barrier


def run_train(args, rank, world, local_rank, dev):
    """configs 2 and 4: the train step.  Config 4 adds the augmented, device-resident training set and the per-step
    device gather of fit() (models_att.py:200) inside the timed region."""
    import torch
    import torch.distributed as dist
    from lcn_pose_b200 import dist as lcn_dist
    from lcn_pose_b200.tools import data as D
    cfg_id = args.config
    c = CONFIGS[cfg_id]
    BATCH, LAYERS, F = c["batch"], c["layers"], c["F"]
    nnz = nnz_of(c["mask"], c["knn"])
    fwd_flop = fwd_flop_per_pose(nnz, LAYERS, F)
    eng = make_engine(cfg_id, args.path, local_rank)
    mode = args.dp_mode
    if world > 1 and mode in ("p2p", "p2p-end"):
        lcn_dist.init_native_dp(eng)
        eng.dp_enable(1 if mode == "p2p" else 2)
    x, y = synth_xy(BATCH, seed=1234 + rank)
    xd, yd = torch.as_tensor(x).to(dev), torch.as_tensor(y).to(dev)
    x_pin, y_pin = torch.as_tensor(x).pin_memory(), torch.as_tensor(y).pin_memory()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)     # > 126 MB L2
    n_bn = 1 + 2 * LAYERS
    barrier = barrier_fn(world)
    gather = None
    if cfg_id == 4:
        # base + flip + rotate(theta) + translate(t) applied identically to inputs (k = 2) and labels (k = 3), one
        # theta ~ U(-60, 60) and t ~ U(-0.1, 0.1) from the recorded seed (SURVEY section 10): 4x the base set, built
        # ON THE DEVICE by lcn_augment, outside the timed region like the reference's one-off host preprocessing
        base_n = 1 << 18
        bx, by = synth_xy(base_n, seed=777 + rank)
        bxd, byd = torch.as_tensor(bx).to(dev), torch.as_tensor(by).to(dev)
        r = np.random.default_rng(2019)
        theta, tr = float(r.uniform(-60, 60)), float(r.uniform(-0.1, 0.1))
        set_x = torch.cat([bxd, D.flip_data(bxd), D.rotate_data(bxd, theta), D.translation_data(bxd, tr)])
        set_y = torch.cat([byd, D.flip_data(byd), D.rotate_data(byd, theta), D.translation_data(byd, tr)])
        gen = torch.Generator(device=dev).manual_seed(99 + rank)
        idx_pool = [torch.randint(0, set_x.shape[0], (BATCH,), device=dev, generator=gen) for _ in range(8)]
        counter = [0]

        def gather(xx, yy):
            eng.gather_rows(set_x, xx, idx_pool[counter[0] % 8], set_y, yy)
            counter[0] += 1

    def step(xx, yy):
        if gather is not None:
            gather(xx, yy)
        if mode == "none":
            return eng.train_step_graph(xx, yy, args.dropout)
        return lcn_dist.dp_train_step(eng, xx, yy, args.dropout, mode=mode, graph=not args.no_graph)

    for _ in range(max(args.warmup, 3)):
        step(xd, yd)
    barrier()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    # ---- device-resident timing: K steps, L2 flushed between steps, CUDA events per step ----
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    for a, b in evs:
        flush.zero_()
        a.record()
        loss, lr = step(xd, yd)
        b.record()
    barrier()
    dev_ms = sum(a.elapsed_time(b) for a, b in evs)
    if args.dump_outputs and rank == 0:
        # what the caller of the last timed step receives (loss, learning rate) and the parameters it leaves behind
        dump_outputs(args.dump_outputs, {"loss": loss.cpu().numpy(), "lr": np.array([lr]), "params": eng.params.cpu().numpy()})
    # ---- end to end through the public API: every step copies ITS inputs from pinned host memory to the device,
    # runs the step and reads the loss back into pinned host memory.  The input copy of step i+1 runs on a copy
    # stream into the other of two device buffers while step i computes (what an input pipeline does); the host
    # waits for the GPU once, after the last loss has landed. ----
    main_s = torch.cuda.current_stream()
    copy_s = torch.cuda.Stream(device=dev)
    bufs = [(torch.empty_like(xd), torch.empty_like(yd)), (torch.empty_like(xd), torch.empty_like(yd))]
    losses_pin = torch.zeros(args.steps).pin_memory()
    copied = [torch.cuda.Event(), torch.cuda.Event()]
    consumed = [torch.cuda.Event(), torch.cuda.Event()]
    for b in range(2):                               # graph capture / warm-up of both buffer sets, untimed
        bufs[b][0].copy_(x_pin); bufs[b][1].copy_(y_pin)
        step(*bufs[b])
        consumed[b].record(main_s)
    barrier()
    t0 = time.perf_counter()
    for i in range(args.steps):
        b = i & 1
        with torch.cuda.stream(copy_s):
            copy_s.wait_event(consumed[b])           # the step that last read this buffer pair has finished
            bufs[b][0].copy_(x_pin, non_blocking=True)
            bufs[b][1].copy_(y_pin, non_blocking=True)
            copied[b].record(copy_s)
        main_s.wait_event(copied[b])
        step(*bufs[b])
        consumed[b].record(main_s)
        losses_pin[i:i + 1].copy_(eng.loss_dev, non_blocking=True)
    barrier()
    e2e_s = time.perf_counter() - t0
    assert bool(torch.isfinite(losses_pin).all()), "non-finite loss in the end-to-end loop"
    # ---- dominant kernel alone: forward mid-layer GEMM (block-sparse X*(W.M)) ----
    import ctypes as C
    from lcn_pose_b200 import _lib as L
    gemm_ms = None
    if rank == 0:
        st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        reps = 20
        call = lambda: L.check(eng.lib.lcn_layer_gemm(eng.h, eng.params.data_ptr(), eng.ws.data_ptr(), eng.ws.numel(), BATCH, BATCH, 2, 0, st))
        for _ in range(3):
            call()
        ge = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
        for a, b in ge:
            flush.zero_()
            a.record()
            call()
            b.record()
        torch.cuda.synchronize()
        gemm_ms = sum(a.elapsed_time(b) for a, b in ge) / reps
    if sampler:
        sampler.stop_flag = True
        sampler.join(timeout=2)
    # ---- BASELINE.json configs[2] shape as a secondary object: fused inference at BN group 256 + Protocol-1/2 evaluation
    # on poses resident in HBM (the end-to-end version from pinned host memory is `--config 3`) ----
    inf = None
    if args.infer_poses > 0 and cfg_id == 2:
        inf = infer_resident(args, rank, world, local_rank, dev, barrier)
    t = torch.tensor([dev_ms, e2e_s] + (inf[1:] if inf else [0, 0, 0]), dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, e2e_s, f_ms, p1_ms, p2_ms = t.tolist()
    eng.close()                  # graphs first, then the handle (and its communicator)
    if rank != 0:
        return None
    tf_burst, tf_sust, hbm, how = measured_peaks()
    value = world * BATCH * args.steps / (dev_ms * 1e-3)
    mult = 3 if args.path == "x3" else 1          # split-bf16 path: three tensor-core products per algorithmic one
    gemm_flop = 2.0 * nnz * F * F * BATCH
    ach = gemm_flop / (gemm_ms * 1e-3) / 1e12
    line = {"metric": "poses/sec (LCN train step)", "value": value, "unit": "poses/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": dev_ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": {"bf16": "bf16", "x3": "bf16x3 (split-bf16 operands, fp32 accumulate: fp32-parity path)", "fp32": "f32"}[args.path],
            "data": "synthetic", "config": workload_config(cfg_id, args.dropout),
            "detail": {"path": args.path, "launch": "eager" if args.no_graph else "cuda-graph replay (one graph per step)",
                       "parallelism": (f"dp{world}: per-GPU BatchNorm statistics; gradient exchange: " +
                                       {"p2p": "two-shot all-reduce over NVLink peer memory inside lcn_model_backward (csrc/lcn_dp.cu), streamed per layer behind the weight-gradient GEMMs, one graph per step",
                                        "p2p-end": "two-shot all-reduce of the whole bucket over NVLink peer memory at the end of lcn_model_backward (csrc/lcn_dp.cu), one graph per step",
                                        "packed": "one torch.distributed all-reduce of the packed bucket between two graphs",
                                        "none": "none (replicas diverge: measurement floor only)"}[mode])
                       if world > 1 else "single GPU"},
            "e2e": {"value": world * BATCH * args.steps / e2e_s, "unit": "poses/s",
                    "h2d_bytes_per_step": int(x_pin.numel() * 4 + y_pin.numel() * 4), "d2h_bytes_per_step": 4},
            "gpu_launches": launches_per_step(n_bn, args.path, gather is not None) * args.steps,
            "step_tensor_frac": value / world * 3 * fwd_flop / (tf_sust * 1e12),
            "roofline": {"bound": "tensor", "kernel": f"mid-layer forward GEMM (block-sparse, {nnz} nonzero {F}x{F} blocks)",
                         "achieved": ach, "peak": tf_burst, "unit": "TFLOP/s", "frac": ach / tf_burst,
                         "tensor_core_flop_multiplier": mult,
                         "traffic": ncu_traffic() if (cfg_id == 2 and args.path == "bf16") else None,
                         "peak_source": how, "ms_per_launch": gemm_ms},
            "clocks": sampler.summary() if sampler else None}
    if inf is not None:
        n_inf = inf[0]
        tot = world * n_inf
        line["inference"] = {
            "workload": f"configs[2] shape: inference at BN group 256 + Protocol-1/2 evaluation, {n_inf} synthetic poses per GPU "
                        f"resident in HBM, sharded by BN group, no collective",
            "forward_poses_per_s": tot / (f_ms * 1e-3),
            "forward_tensor_frac_burst": n_inf / (f_ms * 1e-3) * fwd_flop / (tf_burst * 1e12),
            "eval_p1_poses_per_s": tot / (p1_ms * 1e-3), "eval_p1_hbm_frac": n_inf * 444 / (p1_ms * 1e-3) / (hbm * 1e9),
            "eval_p2_poses_per_s": tot / (p2_ms * 1e-3), "eval_p2_hbm_frac": n_inf * 444 / (p2_ms * 1e-3) / (hbm * 1e9)}
    # CPU baseline: bounded sample on this box's host cores (rank 0, N=1 only), same batch / dropout / model
    if world == 1 and not args.no_cpu_baseline:
        cs = 6
        dt, threads, cb = cpu_train_steps(cfg_id, args.dropout, cs, 1)
        line["cpu_baseline"] = {"value": cb * cs / dt, "unit": "poses/s", "cores": threads, "kind": "port",
                                "sample": f"{cs} train steps at batch {cb}, dropout {args.dropout}: dense fp32 restatement of the "
                                          f"TF graph (torch-CPU autograd + TF1 Adam); TensorFlow 2.13 not installable offline"}
    return line


def infer_resident(args, rank, world, local_rank, dev, barrier):
    import torch
    from lcn_pose_b200.engine import eval_mpjpe
    n_inf = (args.infer_poses // 256) * 256
    eng2 = make_engine(2, args.path if args.path != "fp32" else "bf16", local_rank)
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    xi = torch.rand((n_inf, 34), device=dev, generator=gen) - 0.5
    oi = torch.empty((n_inf, 51), device=dev)
    gt = torch.randn((n_inf, 17, 3), device=dev, generator=gen) * 300 + torch.tensor([0., 0., 4500.], device=dev)
    box = torch.tensor([0., 0., 999., 999.], device=dev).repeat(n_inf, 1)
    cam = torch.tensor([1145.05, 1143.78, 512.54, 515.45], device=dev).repeat(n_inf, 1)
    rd = gt[:, 0, 2].contiguous()

    def best_ms(fn, reps=3):
        fn()
        barrier()
        evs2 = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
        for a, b in evs2:
            a.record(); fn(); b.record()
        barrier()
        return min(a.elapsed_time(b) for a, b in evs2)
    f_ms = best_ms(lambda: eng2.forward(xi, bn_group=256, out=oi))
    pred = oi.view(n_inf, 17, 3)
    p1_ms = best_ms(lambda: eval_mpjpe(pred, gt, box, cam, rd, False, want_err=False))
    p2_ms = best_ms(lambda: eval_mpjpe(pred, gt, box, cam, rd, True, want_err=False))
    return [n_inf, f_ms, p1_ms, p2_ms]


def run_config3(args, rank, world, local_rank, dev):
    """BASELINE.json configs[2] as ONE measured pipeline, end to end from pinned host memory: per chunk H2D of the 2D
    inputs and of the evaluation side data (gt, box, camera, root depth), inference at BatchNorm group 256 (fused stack
    kernel), DataReader.denormalize, Protocol-1 AND Protocol-2 evaluation into fp64 sums on the device -- no host hop
    between the stages (the reference goes through result.pkl, inference.py:113-120 -> evaluate.py:30-45).  The pose set
    is sharded over the ranks by BatchNorm group, no collective on the data path, one all-reduce of the [19] sums."""
    import ctypes as C
    import torch
    import torch.distributed as dist
    from lcn_pose_b200 import _lib as L
    from lcn_pose_b200 import dist as lcn_dist
    from lcn_pose_b200.engine import eval_mpjpe
    total = args.total_poses
    lo, hi = lcn_dist.shard_groups(total, 256, rank, world)
    n_mine = hi - lo
    chunk = 1 << 20
    eng = make_engine(3, args.path if args.path != "fp32" else "bf16", local_rank)
    eng.reserve_ws((chunk, 256, False))
    eng.prepare()
    # a pool of pinned host chunks stands in for the dataset (H36M-shaped synthetic, SURVEY 8(d)); every chunk of the
    # shard is copied from it inside the timed region
    rng = np.random.default_rng(1234 + rank)
    pool = 2
    host = []
    for _ in range(pool):
        x2d = torch.from_numpy((rng.random((chunk, 34), dtype=np.float32) - 0.5)).pin_memory()
        gt = torch.from_numpy((rng.standard_normal((chunk, 51), dtype=np.float32) * 300)).pin_memory()
        gt.view(chunk, 17, 3)[:, :, 2] += 4500.0
        side = torch.empty((chunk, 11), dtype=torch.float32)            # box 4, cam 4, root depth 1, res 2
        side[:, 0:4] = torch.tensor([0., 0., 999., 999.])
        side[:, 4:8] = torch.tensor([1145.05, 1143.78, 512.54, 515.45])
        side[:, 8] = gt.view(chunk, 17, 3)[:, 0, 2]
        side[:, 9:11] = torch.tensor([1000., 1002.])
        host.append((x2d, gt, side.pin_memory()))
    bufs = [tuple(torch.empty_like(t, device=dev) for t in host[0]) for _ in range(2)]
    outs = [torch.empty((chunk, 51), device=dev) for _ in range(2)]
    box = [torch.empty((chunk, 4), device=dev) for _ in range(2)]
    cam = [torch.empty((chunk, 4), device=dev) for _ in range(2)]
    rd = [torch.empty((chunk,), device=dev) for _ in range(2)]
    res = [torch.empty((chunk, 2), device=dev) for _ in range(2)]
    sums = torch.zeros((2, 1, 19), dtype=torch.float64, device=dev)
    main_s, copy_s = torch.cuda.current_stream(), torch.cuda.Stream(device=dev)
    copied, consumed = [torch.cuda.Event(), torch.cuda.Event()], [torch.cuda.Event(), torch.cuda.Event()]
    barrier = barrier_fn(world)
    lib = L.load()

    def run(n_poses, timed):
        sums.zero_()
        done = 0
        i = 0
        while done < n_poses:
            m = min(chunk, n_poses - done)
            b = i & 1
            hx, hg, hs = host[i % pool]
            with torch.cuda.stream(copy_s):
                if i >= 2:
                    copy_s.wait_event(consumed[b])
                bufs[b][0][:m].copy_(hx[:m], non_blocking=True)
                bufs[b][1][:m].copy_(hg[:m], non_blocking=True)
                bufs[b][2][:m].copy_(hs[:m], non_blocking=True)
                copied[b].record(copy_s)
            main_s.wait_event(copied[b])
            side = bufs[b][2]
            box[b][:m].copy_(side[:m, 0:4]); cam[b][:m].copy_(side[:m, 4:8]); rd[b][:m].copy_(side[:m, 8]); res[b][:m].copy_(side[:m, 9:11])
            eng.forward(bufs[b][0][:m], bn_group=256, training=False, out=outs[b][:m])
            pose = outs[b][:m].view(m, 17, 3)
            L.check(lib.lcn_denormalize(pose.data_ptr(), res[b].data_ptr(), m, C.c_void_p(main_s.cuda_stream)))
            gtd = bufs[b][1][:m].view(m, 17, 3)
            for p2 in (0, 1):
                L.check(lib.lcn_eval_mpjpe(pose.data_ptr(), gtd.data_ptr(), box[b].data_ptr(), cam[b].data_ptr(), rd[b].data_ptr(),
                                           None, 0, m, p2, None, None, sums[p2].data_ptr(), C.c_void_p(main_s.cuda_stream)))
            consumed[b].record(main_s)
            done += m
            i += 1
        s = sums.clone()
        if world > 1:
            lcn_dist.all_reduce_eval_sums(s)
        return s.cpu()          # the D2H read of the result: 2 x 19 doubles

    run(min(n_mine, 2 * chunk), False)          # warm-up (>= 3 forward launches incl. the workspace first touch)
    run(min(n_mine, 2 * chunk), False)
    barrier()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    reps = args.steps
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t0 = time.perf_counter()
    e0.record()
    for _ in range(reps):
        s = run(n_mine, True)
    e1.record()
    barrier()
    wall = time.perf_counter() - t0
    dev_ms = e0.elapsed_time(e1)
    if sampler:
        sampler.stop_flag = True
        sampler.join(timeout=2)
    t = torch.tensor([dev_ms, wall], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, wall = t.tolist()
    if rank != 0:
        return None
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"eval_sums": s.numpy()})
    tf_burst, tf_sust, hbm, how = measured_peaks()
    c = CONFIGS[3]
    fwd_flop = fwd_flop_per_pose(nnz_of(c["mask"], c["knn"]), c["layers"], c["F"])
    value = total * reps / (dev_ms * 1e-3)
    allr = s[:, 0, :]
    return {"metric": "poses/sec (LCN inference + Protocol-1/2 MPJPE evaluation pipeline)", "value": value, "unit": "poses/s",
            "n_gpus": world, "steps": reps, "warmup": 2, "ms_per_step": dev_ms / reps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": dict(workload_config(3, 0.0), total_poses=total,
                           l2="inputs (" + str(total // world * 376 // (1 << 20)) + " MiB per GPU and pass) are far larger than the 126 MB L2"),
            "detail": {"path": args.path, "launch": "eager, double-buffered H2D on a copy stream",
                       "parallelism": f"{world} GPU(s): contiguous ranges of BatchNorm groups per rank, no collective on the data path, "
                                      f"one all-reduce of 2 x 19 fp64 sums"},
            "e2e": {"value": total * reps / wall, "unit": "poses/s", "h2d_bytes_per_step": int(n_mine * 376), "d2h_bytes_per_step": 2 * 19 * 8},
            "gpu_launches": reps * ((n_mine + chunk - 1) // chunk) * 4,
            "pipeline_tensor_frac_burst": value / world * fwd_flop / (tf_burst * 1e12),
            "result": {"mpjpe_p1_mm": float(allr[0, :17].sum() / (17 * allr[0, 17])), "mpjpe_p2_mm": float(allr[1, :17].sum() / (17 * allr[1, 17])),
                       "poses_counted": float(allr[0, 17])},
            "roofline": {"bound": "tensor", "kernel": "k_lcn_stack (fused inference, whole pipeline time in the denominator)",
                         "achieved": value / world * fwd_flop / 1e12, "peak": tf_burst, "unit": "TFLOP/s",
                         "frac": value / world * fwd_flop / (tf_burst * 1e12), "traffic": None, "peak_source": how},
            "clocks": sampler.summary() if sampler else None}


def run_config5(args, rank, world, local_rank, dev):
    """BASELINE.json configs[4]: L=5, F=128, batch 16384, knn in {1, 2, 3, full}: train step and mid-layer GEMM against
    mask density.  `value` is the knn=3 train step; the sweep is under `sweep`.  Single GPU."""
    import ctypes as C
    import torch
    from lcn_pose_b200 import _lib as L
    if rank != 0:
        return None
    c = CONFIGS[5]
    B, F, LAYERS = c["batch"], c["F"], c["layers"]
    tf_burst, tf_sust, hbm, how = measured_peaks()
    x, y = synth_xy(B, seed=1234)
    xd, yd = torch.as_tensor(x).to(dev), torch.as_tensor(y).to(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    sweep, head, outputs = [], None, {}
    sampler = ClockSampler(local_rank)
    sampler.start()
    for knn in (1, 2, 3, 17):
        eng = make_engine(5, args.path, local_rank, knn=knn)
        nnz = int((eng.support != 0).sum())
        fwd_flop = fwd_flop_per_pose(nnz, LAYERS, F)
        for _ in range(max(args.warmup, 3)):
            eng.train_step_graph(xd, yd, args.dropout)
        torch.cuda.synchronize()
        reps = args.steps
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
        for a, b in ev:
            flush.zero_()
            a.record(); loss, lr = eng.train_step_graph(xd, yd, args.dropout); b.record()
        torch.cuda.synchronize()
        ms = sum(a.elapsed_time(b) for a, b in ev) / reps
        if args.dump_outputs:
            tag = "full" if knn == 17 else knn
            outputs.update({f"knn{tag}_loss": loss.cpu().numpy(), f"knn{tag}_lr": np.array([lr]),
                            f"knn{tag}_params": eng.params.cpu().numpy()})
        st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        call = lambda: L.check(eng.lib.lcn_layer_gemm(eng.h, eng.params.data_ptr(), eng.ws.data_ptr(), eng.ws.numel(), B, B, 2, 0, st))
        call()
        for a, b in ev:
            flush.zero_()
            a.record(); call(); b.record()
        torch.cuda.synchronize()
        gms = sum(a.elapsed_time(b) for a, b in ev) / reps
        gflop = 2.0 * nnz * F * F * B
        row = {"knn": "full" if knn == 17 else knn, "nnz_blocks_of_289": nnz, "train_ms": ms, "train_poses_per_s": B / ms * 1e3,
               "train_tensor_frac_sustained": B / ms * 1e3 * 3 * fwd_flop / (tf_sust * 1e12), "mid_gemm_ms": gms,
               "mid_gemm_tflops": gflop / gms / 1e9, "mid_gemm_tensor_frac_burst": gflop / gms / 1e9 / tf_burst}
        sweep.append(row)
        if knn == 3:
            head = (row, reps)
        del eng
        torch.cuda.empty_cache()
    sampler.stop_flag = True
    sampler.join(timeout=2)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs)
    row, reps = head
    return {"metric": "poses/sec (LCN train step)", "value": row["train_poses_per_s"], "unit": "poses/s", "n_gpus": 1,
            "steps": reps, "warmup": max(args.warmup, 3), "ms_per_step": row["train_ms"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16" if args.path == "bf16" else args.path, "data": "synthetic",
            "config": workload_config(5, args.dropout), "detail": {"path": args.path, "launch": "cuda-graph replay", "parallelism": "single GPU"},
            "gpu_launches": launches_per_step(1 + 2 * LAYERS, args.path) * reps,
            "roofline": {"bound": "tensor", "kernel": "mid-layer forward GEMM (block-sparse, 175 nonzero 128x128 blocks)",
                         "achieved": row["mid_gemm_tflops"], "peak": tf_burst, "unit": "TFLOP/s",
                         "frac": row["mid_gemm_tensor_frac_burst"], "traffic": None, "peak_source": how, "ms_per_launch": row["mid_gemm_ms"]},
            "sweep": sweep, "clocks": sampler.summary()}


JSON_OUT = sys.stdout


def main():
    if os.environ.get("LCN_HANG_TRACE"):          # debugging aid: dump every thread's Python stack after N seconds
        import faulthandler
        faulthandler.dump_traceback_later(float(os.environ["LCN_HANG_TRACE"]), exit=False)
    # The contract is ONE JSON line on stdout.  NCCL prints its version banner with a C-level printf to stdout when the
    # first communicator is created (seen on the GPU boxes: "NCCL version 2.28.9+cuda12.9" in front of the line), so the
    # process's fd 1 is pointed at stderr and the JSON line goes to a duplicate of the original stdout.
    global JSON_OUT
    sys.stdout.flush()
    JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=sorted(CONFIGS), help="BASELINE.json configs index + 1 (2 = the headline)")
    ap.add_argument("--path", default=os.environ.get("LCN_BENCH_PATH", "bf16"), choices=["bf16", "x3", "fp32"],
                    help="bf16: 1e-2 parity path; x3 (= fp32): fp32-parity path on the tensor cores (split-bf16 operands)")
    ap.add_argument("--dropout", type=float, default=0.25)     # params_help.py:166 training default
    ap.add_argument("--dp-mode", default=os.environ.get("LCN_DP_MODE", "p2p"), choices=["p2p", "p2p-end", "packed", "none"],
                    help="gradient exchange: p2p (library kernel over NVLink peer memory), packed (torch / NCCL all-reduce of the packed "
                         "bucket), none (NO exchange -- calibration of the multi-process overhead only, replicas diverge)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--infer-poses", type=int, default=1 << 22, help="poses per GPU of the secondary resident inference+eval leg (0: skip)")
    ap.add_argument("--total-poses", type=int, default=1 << 26, help="--config 3: poses of the whole job (sharded over the GPUs)")
    ap.add_argument("--no-graph", action="store_true", help="eager launches instead of CUDA-graph replay")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed as DIR/<name>.npy "
                                                          "(float32 / float64, at most 60 MiB in all; rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU arm; --impl reference has none to write")
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_gpu(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
