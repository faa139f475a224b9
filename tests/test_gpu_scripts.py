"""The reference's three scripts against the shims (SURVEY 8(b): "train.py, inference.py and evaluate.py unchanged").

Two tests:
 * test_reference_scripts_run_unmodified -- executes the reference's OWN script source (train.py, inference.py,
   evaluate.py read at test time from the checkout LCN_REFERENCE_DIR names, not copied) with `shims/`
   (+ `shims/optional_stubs/`) in front of sys.path, __file__ relocated to a scratch root so that their `experiment/`
   and `dataset/` live there, and sys.argv set to the flags a user would pass.  Needs BOTH a GPU and a checkout of the
   reference: it is the proof for whoever has both, and skips otherwise.
 * test_script_call_sequences_through_the_shims -- the same module-level calls the three scripts make, in their order
   (cited line by line), on synthetic pickles in the tools/gendb.py:66-81 schema.  Runs on the GPU box.  Checks the
   artefacts the scripts exchange (checkpoints, result.pkl) and the final MPJPE tables against the float64 oracle."""
import contextlib
import importlib
import io
import os
import pickle
import sys
import types

import numpy as np
import pytest
import torch

from oracle import lcn_oracle as O

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("LCN_REFERENCE_DIR")
FX, FY, CX, CY = 1145.05, 1143.78, 512.54, 515.45


def _dataset(n, seed, cams=("54138969", "55011271")):
    """dataitems with the keys tools/gendb.py:66-81 writes (those the path reads)."""
    rng = np.random.default_rng(seed)
    items = []
    for i in range(n):
        root = np.array([rng.normal(0, 500), rng.normal(0, 500), rng.uniform(3000, 6000)])
        j3c = root + rng.normal(0, 300, (17, 3))
        j3c[0] = root
        tl = [(root[0] - 1000) / root[2] * FX + CX, (root[1] - 1000) / root[2] * FY + CY]
        br = [(root[0] + 1000) / root[2] * FX + CX, (root[1] + 1000) / root[2] * FY + CY]
        box = np.array(tl + br)
        ratio = (box[2] - box[0] + 1) / 2000.0
        j3i = np.stack([j3c[:, 0] / j3c[:, 2] * FX + CX, j3c[:, 1] / j3c[:, 2] * FY + CY, (j3c[:, 2] - root[2]) * ratio], 1)
        items.append({"videoid": i // 50, "cameraid": i % 2, "imageid": i,
                      "camera_param": {"name": cams[i % 2], "fx": FX, "fy": FY, "cx": CX, "cy": CY},
                      "joint_3d_image": j3i, "joint_3d_camera": j3c, "box": box, "subject": 1 + i % 3, "action": 2 + i % 4,
                      "subaction": 1, "root_depth": j3c[0, 2]})
    return items


@contextlib.contextmanager
def _shimmed(root):
    saved_path, saved_env = list(sys.path), os.environ.get("LCN_ROOT_PATH")
    stale = [k for k in sys.modules if k in ("tools", "network", "tensorflow", "prettytable") or k.startswith(("tools.", "network."))]
    saved = {k: sys.modules.pop(k) for k in stale}
    sys.path[:0] = [os.path.join(ROOT, "shims"), os.path.join(ROOT, "shims", "optional_stubs")]
    os.environ["LCN_ROOT_PATH"] = root
    try:
        yield
    finally:
        sys.path[:] = saved_path
        for k in [k for k in sys.modules if k in ("tools", "network", "tensorflow", "prettytable") or k.startswith(("tools.", "network."))]:
            del sys.modules[k]
        sys.modules.update(saved)
        if saved_env is None:
            os.environ.pop("LCN_ROOT_PATH", None)
        else:
            os.environ["LCN_ROOT_PATH"] = saved_env


def _write_datasets(root):
    os.makedirs(os.path.join(root, "dataset"), exist_ok=True)
    sets = {"train": _dataset(1200, 1), "val": _dataset(300, 2), "test": _dataset(500, 3)}
    for k, v in sets.items():
        with open(os.path.join(root, "dataset", "h36m_%s.pkl" % k), "wb") as f:
            pickle.dump(v, f)
    os.makedirs(os.path.join(root, "experiment", "test1"), exist_ok=True)
    return sets


@pytest.mark.skipif(not REF, reason="needs a checkout of the reference named by LCN_REFERENCE_DIR")
def test_reference_scripts_run_unmodified(tmp_path):
    root = str(tmp_path)
    _write_datasets(root)

    def run(script, argv):
        src = open(os.path.join(REF, script)).read()                   # read, compiled and executed; never copied
        fake = os.path.join(root, script)
        g = {"__name__": "__main__", "__file__": fake}
        old_argv = sys.argv
        sys.argv = [fake] + argv
        try:
            exec(compile(src, fake, "exec"), g)
        finally:
            sys.argv = old_argv
    with _shimmed(root):
        run("train.py", ["--train_set", "h36m", "--validation_set", "h36m", "--knn", "2", "--layers", "1", "--epochs", "2",
                         "--batch_size", "200", "--flip-data"])
        run("inference.py", ["--train_set", "h36m", "--test_set", "h36m", "--knn", "2", "--layers", "1", "--batch_size", "200",
                             "--dropout", "0", "--checkpoints", "final"])
        run("evaluate.py", ["--filename", "h36m", "--test-indices", "1", "--per-joint"])
        run("evaluate.py", ["--filename", "h36m", "--test-indices", "1", "--protocol2"])
    assert os.path.exists(os.path.join(root, "experiment", "test1", "result.pkl"))
    assert any(f.startswith("err__joint") for f in os.listdir(os.path.join(root, "experiment", "test1")))


def test_script_call_sequences_through_the_shims(tmp_path):
    root = str(tmp_path)
    sets = _write_datasets(root)
    args = types.SimpleNamespace(test_indices="1", mask_type="locally_connected", init_type="same", knn=2, layers=1, dropout=0.0,
                                 channels=64, checkpoints="final", epochs=2, batch_size=200, learning_rate=1e-3,
                                 regularization=None)
    with _shimmed(root), contextlib.redirect_stdout(io.StringIO()):
        data = importlib.import_module("tools.data")
        params_help = importlib.import_module("tools.params_help")
        models_att = importlib.import_module("network.models_att")
        tools = importlib.import_module("tools.tools")
        assert os.path.join(ROOT, "shims") in models_att.__file__
        # ---- train.py:49-113 ----
        datareader = data.DataReader()
        gt_trainset = datareader.real_read("h36m", "train")                       # :53
        gt_valset = datareader.real_read("h36m", "val")                           # :54
        train_data, val_data = datareader.read_2d(gt_trainset, gt_valset)         # :78
        train_labels, val_labels = datareader.read_3d()                           # :79
        dataset_copy, labelset_copy = train_data.copy(), train_labels.copy()
        train_data = np.concatenate((train_data, data.flip_data(dataset_copy)), axis=0)        # :86
        train_labels = np.concatenate((train_labels, data.flip_data(labelset_copy)), axis=0)   # :87
        params = params_help.get_params(is_training=True, gt_dataset=train_labels)             # :107
        params_help.update_parameters(args, params)                               # :108
        network = models_att.cgcnn(**params)                                      # :111
        losses, t_step = network.fit(train_data, train_labels, val_data, val_labels, None, starting_checkpoint=None)   # :113
        assert len(losses) == 2 and t_step > 0 and losses[-1] < losses[0]
        ck = os.path.join(root, "experiment", "test1", "checkpoints", "final")
        assert "checkpoint" in os.listdir(ck)
        # ---- inference.py:53-120, with --flip-data test-time augmentation ----
        datareader = data.DataReader()
        gt_trainset = datareader.real_read("h36m", "train")                       # :56
        gt_testset = datareader.real_read("h36m", "test")                         # :57
        _, test_data = datareader.read_2d(gt_trainset, gt_testset)                # :64
        train_labels, test_labels = datareader.read_3d()                          # :65
        dataset_copy = test_data.copy()
        test_aug = np.concatenate((test_data, data.flip_data(dataset_copy)), axis=0)           # :76
        op_ord, num_aug = {"f": 1}, 1                                             # :78-79
        params = params_help.get_params(is_training=True, gt_dataset=train_labels)             # :99
        params_help.update_parameters(args, params)
        network = models_att.cgcnn(**params)                                      # :104 (a NEW model: restores the checkpoint)
        predictions = network.predict(data=test_aug, sess=None)                   # :106
        assert predictions.shape == (1000, 51) and predictions.dtype == np.float64
        predictions = data.undo(predictions, op_ord, number_actions=num_aug, translation=None)   # :110-111 (translation stays None without --translate_data)
        result = datareader.denormalize(predictions)                              # :113
        with open(os.path.join(root, "experiment", params["dir_name"], "result.pkl"), "wb") as f:   # :114-120
            pickle.dump(result, f)
        # ---- evaluate.py:29-110 (per pose, the reference's loop) on the first poses; evaluate_batch on all ----
        with open(os.path.join(root, "experiment", "test1", "result.pkl"), "rb") as f:
            preds = np.reshape([r["result"] for r in pickle.load(f)], (-1, 17, 3))            # :33-45
        gt_items = sets["test"]
        per_pose = []
        for idx in range(40):
            pred = tools.image_to_camera_frame(pose3d_image_frame=preds[idx], box=gt_items[idx]["box"],
                                               camera=gt_items[idx]["camera_param"], rootIdx=0,
                                               root_depth=gt_items[idx]["root_depth"])        # :54-56
            pred = tools.align_to_gt(pose=pred, pose_gt=gt_items[idx]["joint_3d_camera"])     # :58-59
            per_pose.append(np.sqrt(np.square(pred - gt_items[idx]["joint_3d_camera"]).sum(axis=1)))   # :61
        gts = np.array([it["joint_3d_camera"] for it in gt_items])
        boxes = np.array([it["box"] for it in gt_items])
        cams = np.tile(np.array([FX, FY, CX, CY]), (len(gt_items), 1))
        rds = np.array([it["root_depth"] for it in gt_items])
        acts = np.array([it["action"] - 2 for it in gt_items], dtype=np.int32)
        rep1 = tools.evaluate_batch(preds, gts, boxes, cams, rds, False, actions=acts, n_actions=4)
        rep2 = tools.evaluate_batch(preds, gts, boxes, cams, rds, True, actions=acts, n_actions=4)
        trained = {k: v.astype(np.float64) for k, v in network.engine.get_params().items()}
    # ---- the oracle on the same trained parameters, float64 end to end ----
    cfg = O.LcnConfig(F=64, num_layers=1, neighbour_matrix=O.get_neighbour_matrix_by_hand(knn=2))
    res = np.array([O.camera_resolution(it["camera_param"]["name"]) for it in gt_items], dtype=np.float64)
    x_ref = O.normalize_2d(np.array([it["joint_3d_image"] for it in gt_items]), res[:, 0], res[:, 1])
    p_ref = O.predict(cfg, trained, np.concatenate([x_ref, O.flip_data(x_ref)]), 200)
    p_ref = O.undo(p_ref, {"f": 1}, number_actions=1, translation=0.0)
    den = O.denormalize(p_ref, res[:, 0], res[:, 1])
    e1 = O.eval_errors(den, gts, boxes, cams, rds, False)
    e2 = O.eval_errors(den, gts, boxes, cams, rds, True)
    assert abs(rep1["mpjpe"] - e1.mean()) < 0.1 and abs(rep2["mpjpe"] - e2.mean()) < 0.1          # north_star: 0.1 mm (bf16 path)
    assert np.abs(rep1["per_joint"] - e1.mean(0)).max() < 0.1 and np.abs(rep2["per_joint"] - e2.mean(0)).max() < 0.1
    assert np.abs(np.array(per_pose) - e2[:40]).max() < 0.5                                       # single poses, bf16 predictions
    for a in range(4):
        assert abs(rep1["per_action"][a] - e1[acts == a].mean()) < 0.1
