"""Synchronised BatchNorm under data parallelism, pinned on the CPU (no GPU):
  * the float64 sharded restatement (tests/sharded_oracle.py: pooled moments forward, pooled S1 / S2 backward, mean of
    the per-rank gradients) equals the oracle's loss_and_grads on the concatenated batch for equal shards, and a torch
    autograd restatement of (1/W) sum_r L_r with pooled BatchNorm for unequal shards;
  * the C ABI switch lcn_dp_sync_batch_norm refuses to turn on for a model that is not connected."""
import ctypes as C

import numpy as np
import pytest

from lcn_pose_b200 import _lib as L
from oracle import lcn_oracle as O
from tests.sharded_oracle import loss_and_grads_sharded, torch_reference

F, B = 8, 24


def _setup(mask_type, residual, drop, seed=0):
    cfg = O.LcnConfig(F=F, num_layers=2, mask_type=mask_type, residual=residual,
                      neighbour_matrix=O.get_neighbour_matrix_by_hand(knn=3))
    p = O.init_params(cfg, seed=seed)
    rng = np.random.default_rng(seed + 1)
    for k in p:                     # away from gamma = 1, beta = 0, mask = L
        if k.endswith("gamma") or k.endswith("beta") or k == "mask":
            p[k] = p[k] + rng.normal(0, 0.1, p[k].shape)
    x = rng.normal(0, 0.3, (B, 34))
    y = rng.normal(0, 0.3, (B, 51))
    keep = [rng.uniform(size=(B, 17 * F)) >= drop for _ in range(cfg.n_lin - 1)] if drop > 0 else None
    return cfg, p, x, y, keep


def _split(a, sizes):
    return np.split(a, np.cumsum(sizes)[:-1]) if a is not None else None


def _shard_keep(keep, sizes):
    if keep is None:
        return None
    per_layer = [_split(k, sizes) for k in keep]
    return [[per_layer[l][r] for l in range(len(keep))] for r in range(len(sizes))]


def _rel(a, b):
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-300))


CASES = [(mt, res, drop) for mt in ("locally_connected", "exponential") for res in (True, False) for drop in (0.0, 0.25)]


@pytest.mark.parametrize("world", [2, 4])
@pytest.mark.parametrize("mask_type,residual,drop", CASES)
def test_equal_shards_equal_the_concatenated_batch(world, mask_type, residual, drop):
    cfg, p, x, y, keep = _setup(mask_type, residual, drop)
    sizes = [B // world] * world
    loss, g, _ = loss_and_grads_sharded(cfg, p, _split(x, sizes), _split(y, sizes), _shard_keep(keep, sizes), drop)
    ref_loss, ref = O.loss_and_grads(cfg, p, x, y, drop, keep)
    assert abs(loss - ref_loss) < 1e-10 * ref_loss
    assert set(g) == set(ref)
    for k in ref:
        assert _rel(g[k], ref[k]) < 1e-10, k


@pytest.mark.parametrize("sizes", [[5, 19], [3, 9, 5, 7]])
@pytest.mark.parametrize("mask_type,residual,drop", CASES)
def test_unequal_shards_equal_the_mean_of_the_shard_losses(sizes, mask_type, residual, drop):
    cfg, p, x, y, keep = _setup(mask_type, residual, drop)
    args = (cfg, p, _split(x, sizes), _split(y, sizes), _shard_keep(keep, sizes), drop)
    loss, g, per_rank = loss_and_grads_sharded(*args)
    ref_loss, ref = torch_reference(*args)
    assert abs(loss - ref_loss) < 1e-10 * ref_loss
    assert set(g) == set(ref)
    for k in ref:
        assert _rel(g[k], ref[k]) < 1e-10, k
    # the objective differs from the MSE of the concatenated batch, so the W x factor and the counts are pinned
    _, cat = O.loss_and_grads(cfg, p, x, y, drop, keep)
    assert max(_rel(g[k], cat[k]) for k in cat) > 1e-3
    # gamma / beta gradients are per-rank sums; their mean is the global gradient
    bn = O.bn_names(cfg)[0]
    np.testing.assert_allclose(sum(r[bn + "/beta"] for r in per_rank) / len(sizes), ref[bn + "/beta"], rtol=1e-10, atol=1e-14)


def test_one_shard_is_the_oracle():
    cfg, p, x, y, _ = _setup("locally_connected", True, 0.0)
    loss, g, _ = loss_and_grads_sharded(cfg, p, [x], [y])
    ref_loss, ref = O.loss_and_grads(cfg, p, x, y)
    assert abs(loss - ref_loss) < 1e-12 * ref_loss
    for k in ref:
        assert _rel(g[k], ref[k]) < 1e-12, k


def _model():
    d = L.ModelDesc()
    d.F, d.in_F, d.num_layers, d.mask_kind, d.path = 64, 2, 1, L.LCN_MASK_LOCALLY_CONNECTED, L.LCN_PATH_BF16
    d.residual, d.batch_norm, d.max_norm = 1, 1, 1
    d.support[:] = (O.get_neighbour_matrix_by_hand(knn=3).T != 0).astype(np.float32).reshape(-1).tolist()
    h = C.c_void_p()
    L.check(L.load().lcn_model_create(C.byref(d), C.byref(h)))
    return h


def test_abi_sync_batch_norm_needs_a_connected_model():
    lib = L.load()
    h = _model()
    try:
        assert lib.lcn_dp_sync_batch_norm(h, 1) == -1                   # LCN_EINVAL
        assert b"not connected" in lib.lcn_last_error()
        assert lib.lcn_dp_sync_batch_norm(h, 0) == 0                    # turning it off is always a valid no-op
        assert lib.lcn_dp_sync_batch_norm(None, 0) == -1
    finally:
        lib.lcn_model_destroy(h)
