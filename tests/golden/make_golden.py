"""Generate golden vectors by running the REFERENCE's own NumPy functions.

Needs a checkout of the reference (adgx/lcn-pose), no GPU:

    LCN_REFERENCE_DIR=/path/to/lcn-pose python tests/golden/make_golden.py

Imports tools/params_help.py, tools/filter_hub.py, tools/tools.py, tools/data.py and
network/models_att.get_exponential_matrix from that checkout with tensorflow / matplotlib /
h5py / prettytable stubbed in sys.modules (they are imported at module top but not used by
the functions called here) and writes tests/golden/reference_numpy.npz.
"""
import contextlib
import io
import os
import sys
import types

import numpy as np

REF = os.environ.get("LCN_REFERENCE_DIR")
HERE = os.path.dirname(os.path.abspath(__file__))


class _Stub(types.ModuleType):
    """Module stub: any attribute resolves to a child stub / no-op callable."""
    __path__ = []

    def __getattr__(self, item):
        if item.startswith("__"):
            raise AttributeError(item)
        child = _Stub(self.__name__ + "." + item)
        setattr(self, item, child)
        return child

    def __call__(self, *a, **k):
        return None


def _stub(name):
    m = _Stub(name)
    sys.modules[name] = m
    return m


def import_reference():
    if not REF:
        sys.exit("set LCN_REFERENCE_DIR to a checkout of the reference")
    for n in ["tensorflow", "matplotlib", "matplotlib.pyplot", "mpl_toolkits", "mpl_toolkits.mplot3d",
              "h5py", "prettytable", "cv2"]:
        _stub(n)
    sys.path.insert(0, REF)
    import importlib
    import importlib.util
    # params_help does a bare `import filter_hub`; pre-load it by path (putting REF/tools on
    # sys.path would make `tools` resolve to tools/tools.py instead of the namespace package)
    spec = importlib.util.spec_from_file_location("filter_hub", os.path.join(REF, "tools", "filter_hub.py"))
    fh = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(fh)
    sys.modules["filter_hub"] = fh
    params_help = importlib.import_module("tools.params_help")
    filter_hub = importlib.import_module("tools.filter_hub")
    tools = importlib.import_module("tools.tools")
    data = importlib.import_module("tools.data")
    models_att = importlib.import_module("network.models_att")
    return params_help, filter_hub, tools, data, models_att


def synth_eval(rng, n):
    """H36M-shaped synthetic evaluation inputs (SURVEY 8(d))."""
    fx, fy, cx, cy = 1145.05, 1143.78, 512.54, 515.45
    root = np.stack([rng.normal(0, 500, n), rng.normal(0, 500, n), rng.uniform(3000, 6000, n)], 1)
    gt = root[:, None, :] + rng.normal(0, 300, (n, 17, 3))
    gt[:, 0] = root
    # box: root +- 1000 mm projected (tools/gendb.py:114-128 shape)
    tl = np.stack([(root[:, 0] - 1000) / root[:, 2] * fx + cx, (root[:, 1] - 1000) / root[:, 2] * fy + cy], 1)
    br = np.stack([(root[:, 0] + 1000) / root[:, 2] * fx + cx, (root[:, 1] + 1000) / root[:, 2] * fy + cy], 1)
    box = np.concatenate([tl, br], 1)
    ratio = (box[:, 2] - box[:, 0] + 1) / 2000.0
    # image-frame prediction = projected gt + noise
    pred = np.empty_like(gt)
    pred[:, :, 0] = gt[:, :, 0] / gt[:, :, 2] * fx + cx
    pred[:, :, 1] = gt[:, :, 1] / gt[:, :, 2] * fy + cy
    pred[:, :, 2] = (gt[:, :, 2] - root[:, None, 2]) * ratio[:, None]
    pred += rng.normal(0, 4.0, pred.shape)
    cam = np.tile(np.array([fx, fy, cx, cy]), (n, 1))
    return pred, gt, box, cam, root[:, 2].copy()


def main():
    params_help, filter_hub, tools, data, models_att = import_reference()
    out = {}
    # ---- masks (bit exact) ----
    for knn in range(1, 6):
        out[f"neighbour_knn{knn}"] = params_help.get_neighbour_matrix_by_hand(filter_hub.neighbour_dict_set[0], knn=knn)
    with contextlib.redirect_stdout(io.StringIO()):
        out["exponential"] = models_att.get_exponential_matrix()
    # ---- SURVEY section 4 known-answer inputs ----
    gt = np.arange(51, dtype=np.float64).reshape(17, 3) ** 1.5
    pred = gt[:, ::-1] * 0.9 + np.sin(np.arange(51)).reshape(17, 3) * 7
    d, Z, tf = tools.procrustes(gt.copy(), pred.copy())
    out["ka_proc_d"], out["ka_proc_Z"], out["ka_proc_scale"] = np.float64(d), Z, np.float64(tf["scale"])
    out["ka_proc_R"] = tf["rotation"]
    out["ka_i2c"] = tools.image_to_camera_frame(np.arange(51, dtype=np.float64).reshape(17, 3) * 3 + 100,
                                               box=[200, 150, 800, 750],
                                               camera={"cx": 512, "cy": 515, "fx": 1145, "fy": 1144},
                                               rootIdx=0, root_depth=5000)
    # ---- seeded batch through the reference evaluate.py:53-61 arithmetic ----
    rng = np.random.default_rng(1234)
    n = 96
    pr, g, box, cam, rd = synth_eval(rng, n)
    # make a few hard cases: reflected prediction, large scale error, near-identical
    p1 = np.empty((n, 17)); p2 = np.empty((n, 17)); aligned = np.empty((n, 17, 3)); camf = np.empty((n, 17, 3))
    for i in range(n):
        c = {"fx": cam[i, 0], "fy": cam[i, 1], "cx": cam[i, 2], "cy": cam[i, 3]}
        pc = tools.image_to_camera_frame(pose3d_image_frame=pr[i], box=box[i], camera=c, rootIdx=0, root_depth=rd[i])
        if i % 16 == 5:      # reflected + scaled copy of gt: det(R) = -1 accepted by the reference
            pc = g[i] * np.array([-1.0, 1.0, 1.0]) * 1.7 + 50.0
        camf[i] = pc
        p1[i] = np.sqrt(np.square(pc - g[i]).sum(axis=1))
        al = tools.align_to_gt(pose=pc.copy(), pose_gt=g[i].copy())
        aligned[i] = al
        p2[i] = np.sqrt(np.square(al - g[i]).sum(axis=1))
    out.update(ev_pred=pr, ev_gt=g, ev_box=box, ev_cam=cam, ev_root_depth=rd, ev_camframe=camf,
               ev_err_p1=p1, ev_err_p2=p2, ev_aligned=aligned)
    # ---- augmentations (tools/data.py) ----
    x2 = rng.normal(0, 0.3, (8, 34)); x3 = rng.normal(0, 0.3, (8, 51))
    out.update(aug_x2=x2, aug_x3=x3, aug_flip2=data.flip_data(x2), aug_flip3=data.flip_data(x3),
               aug_rot2=data.rotate_data(x2, 37.0), aug_rot3=data.rotate_data(x3, 37.0),
               aug_tr2=data.translation_data(x2, 0.07), aug_tr3=data.translation_data(x3, 0.07))
    # ---- test-time-augmentation undo (tools/data.py:269-287): original + flip + rotate(180) + translate slices ----
    u_in = rng.normal(0, 0.3, (4 * 6, 51))
    out.update(aug_undo_in=u_in,
               aug_undo_out=data.undo(u_in, {"f": 1, "r": 2, "t": 3}, number_actions=3, angle=180, translation=0.07),
               aug_undo_fr_out=data.undo(u_in[:18], {"r": 1, "f": 2}, number_actions=2, angle=180, translation=0.0))
    # ---- tools.procrustes with every option of its signature (tools/tools.py:96-181) ----
    A = g[:12].copy()
    B = camf[:12].copy()
    B[3] = A[3] * np.array([-1.0, 1.0, 1.0]) * 0.8 + 30.0          # a reflected input: the forced variants differ from 'best'
    for tag, kw in (("best", {}), ("noscale", {"scaling": False}), ("norefl", {"reflection": False}),
                    ("refl", {"reflection": True}), ("noscale_norefl", {"scaling": False, "reflection": False})):
        ds, Zs, Rs, ss, ts = [], [], [], [], []
        for i in range(len(A)):
            d_, Z_, tf_ = tools.procrustes(A[i].copy(), B[i].copy(), **kw)
            ds.append(d_); Zs.append(Z_); Rs.append(tf_["rotation"]); ss.append(tf_["scale"]); ts.append(tf_["translation"])
        out.update({f"proc_{tag}_d": np.array(ds), f"proc_{tag}_Z": np.array(Zs), f"proc_{tag}_R": np.array(Rs),
                    f"proc_{tag}_scale": np.array(ss, dtype=np.float64), f"proc_{tag}_t": np.array(ts)})
    out.update(proc_A=A, proc_B=B)
    # ---- DataReader.read_2d / read_3d / denormalize (tools/data.py:338-489) on a synthetic dataitem list covering the
    # three resolution classes; keys as tools/gendb.py:66-81 writes them ----
    cams = ["54138969", "55011271", "cam_3", "7", "60457274", "58860488"]
    def items(n, seed):
        r = np.random.default_rng(seed)
        return [{"joint_3d_image": np.concatenate([r.uniform(0, 1000, (17, 2)), r.normal(0, 200, (17, 1))], 1),
                 "camera_param": {"name": cams[i % len(cams)]}, "cameraid": i % 4, "videoid": i, "subject": 1 + i % 3,
                 "action": 2 + i % 5} for i in range(n)]
    tr, te = items(7, 1), items(11, 2)
    dr = data.DataReader()
    with contextlib.redirect_stdout(io.StringIO()):
        x_tr, x_te = dr.read_2d(tr, te)
        y_tr, y_te = dr.read_3d()
        res = dr.denormalize(y_te.copy())
    out.update(dr_train_j3d=np.array([it["joint_3d_image"] for it in tr]), dr_test_j3d=np.array([it["joint_3d_image"] for it in te]),
               dr_train_cam=np.array([it["camera_param"]["name"] for it in tr]), dr_test_cam=np.array([it["camera_param"]["name"] for it in te]),
               dr_x_train=x_tr, dr_x_test=x_te, dr_y_train=y_tr, dr_y_test=y_te,
               dr_denorm=np.array([r_["result"] for r_ in res]),
               dr_denorm_action=np.array([r_["action"] for r_ in res]))
    np.savez_compressed(os.path.join(HERE, "reference_numpy.npz"), **out)
    print("wrote", os.path.join(HERE, "reference_numpy.npz"), "with", len(out), "arrays")


if __name__ == "__main__":
    main()
