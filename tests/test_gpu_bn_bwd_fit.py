"""Backward BatchNorm kernels (k_bn_bwd_reduce / k_bn_bwd_apply, lcn_kernels.cu).

They run while the weight-gradient GEMM of the previous layer (k_tc_wgrad) is still on the side stream, and their grid
assumes two blocks per SM: lcn_debug_bn_bwd_fit checks that two blocks of each fit beside one k_tc_wgrad CTA on this
device.  The outputs of the kernels -- dZ, the BatchNorm parameter gradients and the bias gradients that are the row sums
of dZ -- are checked after one CUDA-graph-replayed train step of the benchmarked model (knn=3, L=3, F=64, dropout 0.25)
against float64 autograd of the torch restatement of the reference graph.  dZ of the first layer is the gradient of a
per-row copy of its bias there."""
import ctypes as C

import numpy as np
import pytest
import torch

from lcn_pose_b200 import _lib as L
from oracle import lcn_oracle as O
from oracle import torch_restatement as T
from tests.gpu_helpers import dev, make_pair, rel_err, synth_xy

pytestmark = pytest.mark.gpu
PADDED = 4096          # rows of the workspace layout for both batch sizes below (128-row tiles)


@pytest.mark.parametrize("F", [64, 128])
def test_two_blocks_of_each_kernel_fit_beside_the_weight_gradient_cta(F):
    lib = L.load()
    out = (C.c_int * 6)()
    L.check(lib.lcn_debug_bn_bwd_fit(F, out))
    names = ["reduce<bf16>", "apply<bf16>", "apply<bf16, sync>", "reduce<sp16>", "apply<sp16>", "apply<sp16, sync>"]
    fit = dict(zip(names, out[:]))
    assert all(v >= 2 for v in fit.values()), fit


def _oracle(cfg, p, x, y, rate, keep):
    """float64 loss gradients of every parameter, and dZ of the first layer (the gradient of its bias per row)"""
    tp = T.build_params(p)
    b0 = O.bias_names(cfg)[0]
    tp[b0] = torch.tensor(np.broadcast_to(p[b0], (x.shape[0], p[b0].size)).copy(), dtype=torch.float64,
                          requires_grad=True)
    km = [torch.tensor(k, dtype=torch.float64) for k in keep]
    loss, _ = T.loss_fn(cfg, tp, torch.tensor(x, dtype=torch.float64), torch.tensor(y, dtype=torch.float64), rate, km)
    loss.backward()
    g = {k: v.grad.numpy() for k, v in tp.items()}
    dz0 = g[b0]
    g[b0] = dz0.sum(axis=0)
    return g, dz0


@pytest.mark.parametrize("path,n", [("bf16", 4096), ("fp32", 4096), ("bf16", 4000)],
                         ids=["bf16-4096", "fp32-4096", "bf16-4000-ragged"])
def test_graph_replayed_step_batchnorm_backward_outputs(path, n):
    rate = 0.25
    eng, cfg, p = make_pair(L=3, knn=3, path=path)
    x, y = synth_xy(n)
    xd, yd = dev(x), dev(y)
    keep = [eng.dropout_keep(l, n, rate).cpu().numpy().astype(bool) for l in range(1 + 2 * cfg.num_layers)]
    ref_g, ref_dz0 = _oracle(cfg, p, x.astype(np.float64), y.astype(np.float64), rate, keep)
    before = eng.params.clone()
    eng.train_step_graph(xd, yd, dropout=rate)
    torch.cuda.synchronize()
    dz0 = eng.read_tensor(6, 0, n, n).cpu().numpy()
    # the same workspace read as a PADDED-row batch: its rows n .. PADDED-1 are the tile padding of this step's dZ
    dz0_padded = eng.read_tensor(6, 0, PADDED, PADDED).cpu().numpy()
    stepped = eng.params.clone()
    eng.params.copy_(before)
    eng.prepare()
    g = eng.unflatten(eng.true_grads())
    eng.params.copy_(stepped)
    eng.prepare()

    tol = {"fp32": 2e-3, "bf16": 5e-2}[path]          # the tolerances of test_gpu_real_shapes / test_gpu_parity
    assert np.array_equal(dz0_padded[:n], dz0)
    assert not dz0_padded[n:].any(), "padding rows of dZ must be zero"
    if path == "fp32":
        assert rel_err(dz0, ref_dz0) < tol, ("dZ0", rel_err(dz0, ref_dz0))
    else:
        # Z rounded to bf16 moves a few elements across the LeakyReLU kink, each then off by 0.8 |dy| (a max-norm error of
        # the order of one): dZ as a whole, in the Frobenius norm and its direction
        fro = float(np.linalg.norm(dz0 - ref_dz0) / np.linalg.norm(ref_dz0))
        cos = float((dz0.astype(np.float64) * ref_dz0).sum() / (np.linalg.norm(dz0) * np.linalg.norm(ref_dz0)))
        assert fro < tol and cos > 0.9995, ("dZ0", fro, cos)
    n_bn = 1 + 2 * cfg.num_layers
    names = [b + s for b in O.bn_names(cfg) for s in ("/gamma", "/beta")] + O.bias_names(cfg)[:n_bn]
    for k in names:
        e = rel_err(g[k], ref_g[k])
        assert e < tol, (k, e)
