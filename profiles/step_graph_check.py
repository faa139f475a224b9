"""Records what one captured train step enqueues, so that two builds of liblcn_b200.so can be compared launch for launch.

For every configuration below the script builds a seeded engine and
  * runs one eager step (forward(training) + backward + Adam) and saves its forward output, loss, raw gradient bucket
    and the parameters after Adam as <name>_<tensor>.npy;
  * warms up eagerly as LcnEngine.train_step_graph does, captures prepare + forward(training) + backward + Adam into a
    torch.cuda.CUDAGraph(keep_graph=True) and walks the captured graph with the CUDA driver API (ctypes);
  * writes <name>.json: the multiset of node labels (type, kernel name, grid, block, dynamic shared memory; memset and
    memcpy extents) and the multiset of edges labelled by their end nodes' labels and the edge data (ports, type: the
    programmatic-launch edges of PDL are type 1).
Kernel names are taken with the per-build hash of anonymous namespaces removed.

    LCN_B200_LIB=<lib> python profiles/step_graph_check.py OUT          # all configurations, one directory per build
    python profiles/step_graph_check.py --compare BASE OTHER [BASE2]    # topology equal? output differences

--compare prints, per configuration, whether the topologies are equal and the largest absolute difference of every
saved tensor between BASE and OTHER, next to the same difference between BASE and BASE2 (a second run of the same
build: the BatchNorm sums use fp64 atomics, so two runs of one build differ in the last bits).  Exit code 0 = every
topology equal and no OTHER difference above four times the run-to-run one (one pair of runs samples that spread only
roughly), with a floor of 1e-6 relative to the tensor's scale.
The two-rank configurations run both ranks on device 0 (CUDA IPC within the device, gloo rendezvous), as
tests/dp_sync_bn_worker.py does on a one-GPU machine."""
import collections
import ctypes as C
import glob
import json
import os
import re
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

# name: (path, knn, num_layers, F, batch, mask, dropout)
CONFIGS = {
    "bf16_c2": ("bf16", 3, 3, 64, 4096, "locally_connected", 0.25),
    "fp32_c2": ("fp32", 3, 3, 64, 4096, "locally_connected", 0.25),
    "bf16_exp": ("bf16", 3, 3, 64, 4096, "exponential", 0.25),
    "bf16_l5f128": ("bf16", 3, 5, 128, 16384, "locally_connected", 0.25),
    "fp32_l5f128": ("fp32", 3, 5, 128, 16384, "locally_connected", 0.25),
    "bf16_l0": ("bf16", 3, 0, 64, 4096, "locally_connected", 0.25),
    "fp32_l0": ("fp32", 3, 0, 64, 4096, "locally_connected", 0.25),
}
DP_CONFIG = ("bf16", 3, 3, 64, 2048, "locally_connected", 0.25)     # per rank
DP_MODES = {"dp1": 1, "dp2": 2}

NODE_TYPES = {0: "kernel", 1: "memcpy", 2: "memset", 3: "host", 4: "graph", 5: "empty", 6: "wait_event",
              7: "event_record", 10: "mem_alloc", 11: "mem_free", 12: "batch_mem_op", 13: "conditional"}


class KernelParams(C.Structure):      # CUDA_KERNEL_NODE_PARAMS_v2
    _fields_ = [("func", C.c_void_p), ("grid", C.c_uint * 3), ("block", C.c_uint * 3), ("shmem", C.c_uint),
                ("kernelParams", C.c_void_p), ("extra", C.c_void_p), ("kern", C.c_void_p), ("ctx", C.c_void_p)]


class MemsetParams(C.Structure):      # CUDA_MEMSET_NODE_PARAMS
    _fields_ = [("dst", C.c_uint64), ("pitch", C.c_size_t), ("value", C.c_uint), ("elementSize", C.c_uint),
                ("width", C.c_size_t), ("height", C.c_size_t)]


def _side(p):
    return [(p + "XInBytes", C.c_size_t), (p + "Y", C.c_size_t), (p + "Z", C.c_size_t), (p + "LOD", C.c_size_t),
            (p + "MemoryType", C.c_int), (p + "Host", C.c_void_p), (p + "Device", C.c_uint64), (p + "Array", C.c_void_p),
            (p + "Reserved", C.c_void_p), (p + "Pitch", C.c_size_t), (p + "Height", C.c_size_t)]


class Memcpy3D(C.Structure):          # CUDA_MEMCPY3D
    _fields_ = _side("src") + _side("dst") + [("WidthInBytes", C.c_size_t), ("Height", C.c_size_t), ("Depth", C.c_size_t)]


class EdgeData(C.Structure):          # CUgraphEdgeData
    _fields_ = [("from_port", C.c_ubyte), ("to_port", C.c_ubyte), ("type", C.c_ubyte), ("reserved", C.c_ubyte * 5)]


def graph_topology(graph):
    cu = C.CDLL("libcuda.so.1")

    def ok(r, what):
        if r != 0:
            raise RuntimeError(f"{what} -> CUresult {r}")

    n = C.c_size_t(0)
    ok(cu.cuGraphGetNodes(C.c_void_p(graph), None, C.byref(n)), "cuGraphGetNodes")
    nodes = (C.c_void_p * n.value)()
    ok(cu.cuGraphGetNodes(C.c_void_p(graph), nodes, C.byref(n)), "cuGraphGetNodes")
    labels = {}
    for h in nodes:
        t = C.c_int()
        ok(cu.cuGraphNodeGetType(C.c_void_p(h), C.byref(t)), "cuGraphNodeGetType")
        lab = [NODE_TYPES.get(t.value, str(t.value))]
        if t.value == 0:
            kp = KernelParams()
            ok(cu.cuGraphKernelNodeGetParams_v2(C.c_void_p(h), C.byref(kp)), "cuGraphKernelNodeGetParams")
            name = C.c_char_p()
            if kp.func:
                ok(cu.cuFuncGetName(C.byref(name), C.c_void_p(kp.func)), "cuFuncGetName")
            else:
                ok(cu.cuKernelGetName(C.byref(name), C.c_void_p(kp.kern)), "cuKernelGetName")
            lab += [re.sub(r"_GLOBAL__N__[0-9a-f]+_", "_GLOBAL__N__", name.value.decode()), list(kp.grid),
                    list(kp.block), kp.shmem]
        elif t.value == 2:
            mp = MemsetParams()
            ok(cu.cuGraphMemsetNodeGetParams(C.c_void_p(h), C.byref(mp)), "cuGraphMemsetNodeGetParams")
            lab += [mp.elementSize, mp.width, mp.height, mp.value]
        elif t.value == 1:
            cp = Memcpy3D()
            ok(cu.cuGraphMemcpyNodeGetParams(C.c_void_p(h), C.byref(cp)), "cuGraphMemcpyNodeGetParams")
            lab += [cp.WidthInBytes, cp.Height, cp.Depth, cp.srcPitch, cp.dstPitch, cp.srcMemoryType, cp.dstMemoryType]
        labels[h] = json.dumps(lab)
    m = C.c_size_t(0)
    ok(cu.cuGraphGetEdges_v2(C.c_void_p(graph), None, None, None, C.byref(m)), "cuGraphGetEdges_v2")
    src, dst, data = (C.c_void_p * m.value)(), (C.c_void_p * m.value)(), (EdgeData * m.value)()
    ok(cu.cuGraphGetEdges_v2(C.c_void_p(graph), src, dst, data, C.byref(m)), "cuGraphGetEdges_v2")
    edges = collections.Counter(json.dumps([labels[s], labels[d], [e.from_port, e.to_port, e.type]])
                                for s, d, e in zip(src, dst, data))
    return {"n_nodes": n.value, "n_edges": m.value,
            "nodes": sorted(collections.Counter(labels.values()).items()), "edges": sorted(edges.items())}


def run_config(name, cfg, out_dir, local=0, dp_mode=None):
    import torch
    from lcn_pose_b200 import dist as lcn_dist
    from lcn_pose_b200.engine import LcnEngine
    from oracle import lcn_oracle as O
    from tests.gpu_helpers import synth_xy
    path, knn, num_layers, F, batch, mask, dropout = cfg
    rank = int(os.environ.get("RANK", "0"))
    eng = LcnEngine(F=F, in_F=2, num_layers=num_layers, mask_type=mask,
                    neighbour_matrix=O.get_neighbour_matrix_by_hand(knn=knn), path=path, device=f"cuda:{local}")
    eng.init_params(seed=42)
    if dp_mode is not None:
        lcn_dist.broadcast_parameters(eng.params)
        lcn_dist.init_native_dp(eng, sync_bn=True)
        eng.dp_enable(dp_mode)
    x, y = synth_xy(batch, seed=300 + rank)
    x, y = torch.as_tensor(x).to(eng.device), torch.as_tensor(y).to(eng.device)
    # one eager step
    out = eng.forward(x, bn_group=batch, training=True, dropout=dropout)
    loss = eng.backward(x, y, dropout)
    outputs = {"out": out.cpu().numpy(), "loss": loss.cpu().numpy(), "grads_raw": eng.grads_raw.cpu().numpy()}
    eng.adam()
    outputs["params"] = eng.params.cpu().numpy()
    for k, v in outputs.items():
        np.save(os.path.join(out_dir, f"{name}_{k}.npy"), v)
    # warm-up as train_step_graph does (first-call attribute setup outside the capture), then the capture
    eng._stage_scalars(eng.step + 1)
    side = torch.cuda.Stream(device=eng.device)
    side.wait_stream(torch.cuda.current_stream(eng.device))
    with torch.cuda.stream(side):
        eng.forward(x, bn_group=batch, training=True, dropout=dropout, out=out, dyn=True)
        eng.backward(x, y, dropout)
        eng.adam(dyn=True)
    torch.cuda.current_stream(eng.device).wait_stream(side)
    torch.cuda.synchronize(eng.device)
    g = torch.cuda.CUDAGraph(keep_graph=True)
    with torch.cuda.graph(g):
        eng.prepare()
        eng.forward(x, bn_group=batch, training=True, dropout=dropout, out=out, dyn=True)
        eng.backward(x, y, dropout)
        eng.adam(dyn=True)
    topo = graph_topology(g.raw_cuda_graph())
    with open(os.path.join(out_dir, f"{name}.json"), "w") as f:
        json.dump(topo, f, indent=0)
    print(f"{name}: {topo['n_nodes']} nodes, {topo['n_edges']} edges, loss {float(outputs['loss'][0]):.6f}", flush=True)
    del g
    torch.cuda.synchronize(eng.device)
    return eng


def dp_worker(out_dir):
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(0)
    dist.init_process_group("gloo")
    rank = dist.get_rank()
    for name, mode in DP_MODES.items():
        eng = run_config(f"{name}_rank{rank}", DP_CONFIG, out_dir, dp_mode=mode)
        dist.barrier()
        eng.close()
    dist.barrier()
    dist.destroy_process_group()


def record(out_dir):
    os.makedirs(out_dir, exist_ok=True)
    for name, cfg in CONFIGS.items():
        run_config(name, cfg, out_dir).close()
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
           "127.0.0.1", "--master-port", "29571", os.path.abspath(__file__), "--dp-worker", out_dir]
    subprocess.run(cmd, check=True, timeout=600, cwd=ROOT)


def compare(base, other, base2=None):
    good = True
    for fn in sorted(glob.glob(os.path.join(base, "*.json"))):
        name = os.path.basename(fn)[:-5]
        with open(fn) as f:
            ta = json.load(f)
        with open(os.path.join(other, name + ".json")) as f:
            tb = json.load(f)
        same = ta == tb
        good &= same
        print(f"{name}: topology {'equal' if same else 'DIFFERENT'} ({ta['n_nodes']} nodes, {ta['n_edges']} edges)")
        for k in ("out", "loss", "grads_raw", "params"):
            a = np.load(os.path.join(base, f"{name}_{k}.npy")).astype(np.float64)
            d = float(np.abs(np.load(os.path.join(other, f"{name}_{k}.npy")) - a).max())
            line = f"    {k:9s} max|other - base| {d:.3e}"
            if base2 is not None:
                d2 = float(np.abs(np.load(os.path.join(base2, f"{name}_{k}.npy")) - a).max())
                line += f"   max|base2 - base| {d2:.3e}"
                if d > max(4 * d2, 1e-6 * float(np.abs(a).max())):
                    line += "   ABOVE four times the run-to-run difference"
                    good = False
            print(line)
    print("PASS" if good else "FAIL")
    return good


if __name__ == "__main__":
    if sys.argv[1] == "--compare":
        sys.exit(0 if compare(*sys.argv[2:5]) else 1)
    elif sys.argv[1] == "--dp-worker":
        dp_worker(sys.argv[2])
    else:
        record(sys.argv[1])
