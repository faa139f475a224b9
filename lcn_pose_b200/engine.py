"""LcnEngine: owns the device buffers (through torch) of one LCN model and drives the C ABI.

torch is plumbing here (device memory, streams, pinned host buffers, torch.distributed); every
arithmetic step of the hot path is a kernel of liblcn_b200.so.
"""
import ctypes as C
import math

import numpy as np
import torch

from . import _lib as L

J = 17


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


class LcnEngine:
    """One model (mask support + layer stack) on one GPU.

    Mirrors the arithmetic of cgcnn (network/models_att.py:475-775) and base_model's loss / Adam
    (:352-421).  `path` selects the arithmetic, both on the tcgen05 tensor cores: "bf16" (bf16 operands, 1e-2 parity)
    or "fp32" (alias "x3": split-bf16 operands, three products per block, fp32 parity -- the 1e-4 path)."""

    def __init__(self, F=64, in_F=2, num_layers=3, mask_type="locally_connected", neighbour_matrix=None,
                 residual=True, batch_norm=True, max_norm=True, path="bf16", device="cuda:0",
                 learning_rate=1e-3, decay_steps=32000, decay_rate=0.96, regularization=0.0):
        if not torch.cuda.is_available():
            raise L.LcnError("LcnEngine needs a CUDA device; there is no CPU fallback")
        self.lib = L.load()
        self.device = torch.device(device)
        torch.cuda.set_device(self.device)
        self.F, self.in_F, self.num_layers = int(F), int(in_F), int(num_layers)
        self.mask_type = mask_type
        if path not in ("bf16", "fp32", "x3"):
            raise ValueError("path must be 'bf16' or 'fp32' (alias 'x3')")
        path = "fp32" if path == "x3" else path
        self.path = path
        desc = L.ModelDesc()
        desc.F, desc.in_F, desc.num_layers = self.F, self.in_F, self.num_layers
        desc.residual, desc.batch_norm, desc.max_norm = int(bool(residual)), int(bool(batch_norm)), int(bool(max_norm))
        desc.path = L.LCN_PATH_BF16 if path == "bf16" else L.LCN_PATH_FP32
        if "exponential" in mask_type:                      # models_att.py:573-574
            em = L.exponential_matrix()
            desc.mask_kind = L.LCN_MASK_CONSTANT
            sup = (em != 0).astype(np.float32)
            cm = em
        else:                                               # models_att.py:547-571
            assert neighbour_matrix is not None
            nm = np.asarray(neighbour_matrix, dtype=np.float32)
            assert nm.shape == (J, J)
            desc.mask_kind = L.LCN_MASK_LOCALLY_CONNECTED
            sup = (nm.T != 0).astype(np.float32)
            cm = np.zeros((J, J), np.float32)
            self.mask_init = nm.T.copy()                    # L = neighbour_matrix.T is the initial value (:549-566)
        self.support = sup.copy()
        desc.support[:] = sup.reshape(-1).tolist()
        desc.const_mask[:] = cm.reshape(-1).tolist()
        h = C.c_void_p()
        L.check(self.lib.lcn_model_create(C.byref(desc), C.byref(h)))
        self.h = h
        self.n_params = int(self.lib.lcn_model_param_count(h))
        self.tensors = {}
        name = C.create_string_buffer(256)
        off, rows, cols = C.c_int64(), C.c_int32(), C.c_int32()
        for i in range(self.lib.lcn_model_num_tensors(h)):
            L.check(self.lib.lcn_model_tensor_info(h, i, name, 256, C.byref(off), C.byref(rows), C.byref(cols)))
            self.tensors[name.value.decode()] = (off.value, rows.value, cols.value)
        self.params = torch.zeros(self.n_params, dtype=torch.float32, device=self.device)
        self.adam_m = torch.zeros_like(self.params)
        self.adam_v = torch.zeros_like(self.params)
        self.grads_raw = torch.zeros_like(self.params)
        self.loss_dev = torch.zeros(1, dtype=torch.float32, device=self.device)
        # op_loss_average state (models_att.py:370-379): [biased EMA of the total loss, steps], updated on the device
        self.ema_dev = torch.zeros(2, dtype=torch.float32, device=self.device)
        self.reg_dev = torch.zeros(1, dtype=torch.float32, device=self.device)       # sum of l2_loss(w*, b*)
        self._reg_scratch = torch.zeros(16, dtype=torch.uint8, device=self.device)
        self.ws = None
        self.learning_rate, self.decay_steps, self.decay_rate = learning_rate, decay_steps, decay_rate
        self.regularization = 0.0 if regularization is None else float(regularization)
        self.step = 0                      # Adam t / global_step
        self.seed = 2019
        self._prepared = False
        self._fwd_geom = None
        # device-resident step scalars (lcn_step_scalars: uint64 step, float lr_t, float reserved) + pinned staging
        self.dyn_dev = torch.zeros(16, dtype=torch.uint8, device=self.device)
        self.dyn_pin = torch.zeros((64, 16), dtype=torch.uint8).pin_memory()   # ring: the host runs ahead of the GPU
        self._dyn_ev = [None] * 64
        self._graphs = {}

    def close(self):
        """Release the model handle.  Captured train-step graphs go first: a CUDA graph that recorded collectives of the
        model's NCCL communicator (data-parallel steps) keeps that communicator referenced, and NCCL does not let go of a
        communicator before every such graph is destroyed -- lcn_model_destroy would wait forever."""
        try:
            if getattr(self, "_graphs", None):
                self._graphs.clear()
                torch.cuda.synchronize(self.device)
        except Exception:
            pass
        try:
            if getattr(self, "h", None):
                if getattr(self, "_dp_bucket_owner", None) is not None:
                    self.grads_raw = None          # a view of the library's peer-mapped bucket, freed with the handle
                    self._dp_bucket_owner = None
                self.lib.lcn_model_destroy(self.h)
                self.h = None
        except Exception:
            pass

    def __del__(self):
        self.close()

    # ---- parameters -------------------------------------------------------------------------
    def tensor(self, name):
        off, rows, cols = self.tensors[name]
        v = self.params[off: off + rows * cols]
        return v.view(rows, cols) if rows > 1 else v

    def _view(self, flat, name):
        off, rows, cols = self.tensors[name]
        v = flat[off: off + rows * cols]
        return v.view(rows, cols) if rows > 1 else v

    def set_params(self, np_params):
        """np_params: dict name -> ndarray, names as in the reference's TF variables."""
        for k, v in np_params.items():
            t = self.tensor(k)
            t.copy_(torch.as_tensor(np.asarray(v, dtype=np.float32).reshape(tuple(t.shape))))
        self._prepared = False

    def get_params(self):
        p = self.params.detach().cpu().numpy()
        return {k: p[o: o + r * c].reshape((r, c) if r > 1 else (c,)).copy() for k, (o, r, c) in self.tensors.items()}

    def unflatten(self, flat):
        f = flat.detach().cpu().numpy()
        return {k: f[o: o + r * c].reshape((r, c) if r > 1 else (c,)).copy() for k, (o, r, c) in self.tensors.items()}

    def init_params(self, seed=42):
        """Reference initialisation (models_att.py:614-628 kaiming for w* and b*, BN gamma=1 beta=0,
        mask var = L, :549-566)."""
        rng = np.random.default_rng(seed)

        def tn(shape):
            out = rng.standard_normal(shape)
            bad = np.abs(out) > 2
            while bad.any():
                out[bad] = rng.standard_normal(int(bad.sum()))
                bad = np.abs(out) > 2
            return out
        p = {}
        for k, (o, r, c) in self.tensors.items():
            base = k.rsplit("/", 1)[-1]
            if k == "mask":
                p[k] = self.mask_init.copy()                # the VALUES of L, not only its zero pattern
            elif base == "gamma":
                p[k] = np.ones(c)
            elif base == "beta":
                p[k] = np.zeros(c)
            elif base.startswith("w"):
                p[k] = tn((r, c)) * math.sqrt(2.0 / r)
            else:
                p[k] = tn((c,)) * math.sqrt(2.0 / c)
        self.set_params(p)
        self.adam_m.zero_()
        self.adam_v.zero_()
        self.step = 0

    # ---- workspace ----------------------------------------------------------------------------
    def _ensure_ws(self, n_rows, bn_group, training):
        need = int(self.lib.lcn_model_workspace_bytes(self.h, n_rows, bn_group, int(training)))
        if need == 0:
            raise L.LcnError(self.lib.lcn_last_error().decode())
        if self.ws is None or self.ws.numel() < need:
            self._realloc_ws(need)
        return self.ws.numel()

    def _realloc_ws(self, need):
        # Captured train-step graphs hold the old blob's address and the packed weights live in its head: a
        # reallocation drops both (they are rebuilt on the next call).  fit() avoids the reallocation altogether by
        # reserving the maximum of its train and predict layouts up front (reserve_ws).
        if self._graphs:
            torch.cuda.synchronize(self.device)
        self._graphs.clear()
        self.ws = torch.empty(need, dtype=torch.uint8, device=self.device)
        self._prepared = False

    def reserve_ws(self, *layouts):
        """Size the workspace once for several (n_rows, bn_group, training) layouts, so that none of them reallocates
        later."""
        need = 0
        for n_rows, bn_group, training in layouts:
            b = int(self.lib.lcn_model_workspace_bytes(self.h, int(n_rows), int(bn_group), int(training)))
            if b == 0:
                raise L.LcnError(self.lib.lcn_last_error().decode())
            need = max(need, b)
        if self.ws is None or self.ws.numel() < need:
            self._realloc_ws(need)
        return self.ws.numel()

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def prepare(self):
        """clip_by_norm + mask_weights + pack for every layer (models_att.py:576-586,659-660)."""
        if self.ws is None:
            self._ensure_ws(128, 128, False)
        L.check(self.lib.lcn_model_prepare_weights(self.h, _ptr(self.params), _ptr(self.ws), self.ws.numel(), self._stream()))
        self._prepared = True

    # ---- forward / train ------------------------------------------------------------------------
    def forward(self, x, bn_group=None, training=False, dropout=0.0, out=None, dyn=False):
        """x: [n, 17*in_F] float32 CUDA tensor.  Returns [n, 51] float32 (models_att.py:707-775).
        dyn=True: the dropout step counter is read from self.dyn_dev on the device (CUDA-graph replay)."""
        assert x.is_cuda and x.dtype == torch.float32 and x.is_contiguous()
        n = x.shape[0]
        bn_group = n if bn_group is None else int(bn_group)
        size = self._ensure_ws(n, bn_group, training)
        if not self._prepared:
            self.prepare()
        if out is None:
            out = torch.empty((n, J * 3), dtype=torch.float32, device=self.device)
        L.check(self.lib.lcn_model_forward(self.h, _ptr(self.params), _ptr(self.ws), size, _ptr(x), n, bn_group,
                                           int(training), float(dropout), self.seed, self.step + 1, _ptr(out),
                                           _ptr(self.dyn_dev) if dyn else C.c_void_p(0), self._stream()))
        self._fwd_geom = (n, bn_group, bool(training))
        return out

    def forward_taps(self, x, bn_group):
        """Inference through the fused cluster kernel with the parity tap: returns (out [n,51] float32,
        taps float32 [n_bn, groups*bn_group, 17*F]) -- every layer output A_l decoded from the kernel's tile layout."""
        n = x.shape[0]
        size = self._ensure_ws(n, bn_group, False)
        if not self._prepared:
            self.prepare()
        n_bn = 1 + 2 * self.num_layers
        tpg = (bn_group + 127) // 128
        groups = (n + bn_group - 1) // bn_group
        tiles = groups * tpg
        taps = torch.zeros((n_bn, tiles, J, 128, 8, 8), dtype=torch.bfloat16, device=self.device)
        out = torch.empty((n, J * 3), dtype=torch.float32, device=self.device)
        L.check(self.lib.lcn_model_forward_taps(self.h, _ptr(self.params), _ptr(self.ws), size, _ptr(x), n, bn_group,
                                                _ptr(out), _ptr(taps), taps.numel() * 2, self._stream()))
        # undo the 128-byte swizzle: stored chunk index = c ^ (r & 7)
        r = torch.arange(128, device=self.device).view(128, 1)
        c = torch.arange(8, device=self.device).view(1, 8)
        src = (c ^ (r & 7)).view(1, 1, 1, 128, 8, 1).expand(n_bn, tiles, J, 128, 8, 8)
        dec = torch.gather(taps, 4, src).float()                       # [n_bn, tiles, 17, 128, 8, 8] logical chunk order
        dec = dec.view(n_bn, groups, tpg, J, 128, 64).permute(0, 1, 2, 4, 3, 5).reshape(n_bn, groups, tpg * 128, J * 64)
        return out, dec[:, :, :bn_group, :].reshape(n_bn, groups * bn_group, J * 64)

    def lr_at(self, step):
        """exponential_decay with global_step = step-1 (models_att.py:386-399)."""
        return self.learning_rate * self.decay_rate ** ((step - 1) / self.decay_steps)

    def backward(self, x, labels, dropout=0.0):
        n = x.shape[0]
        assert self._fwd_geom == (n, n, True), "backward needs forward(training=True) with one BN group"
        L.check(self.lib.lcn_model_backward(self.h, _ptr(self.params), _ptr(self.ws), self.ws.numel(), _ptr(x),
                                            _ptr(labels), n, float(dropout), self.seed, self.step + 1,
                                            _ptr(self.loss_dev), _ptr(self.grads_raw), self._stream()))
        return self.loss_dev

    # ---- data-parallel exchange inside the backward pass (csrc/lcn_dp.cu) ---------------------------------
    def dp_export(self, world):
        """Allocate this rank's exchange buffer and return its 64-byte CUDA IPC handle (lcn_dp_export)."""
        buf = (C.c_uint8 * 64)()
        L.check(self.lib.lcn_dp_export(self.h, int(world), C.byref(buf)))
        return bytes(buf)

    def dp_connect(self, handles, rank, world):
        """Map every rank's exchange buffer (lcn_dp_connect).  handles: the `world` handles of dp_export in rank order.
        From here on backward() returns rank-averaged gradients."""
        blob = b"".join(bytes(h) for h in handles)
        assert len(blob) == 64 * world
        buf = (C.c_uint8 * len(blob)).from_buffer_copy(blob)
        L.check(self.lib.lcn_dp_connect(self.h, C.byref(buf), int(rank), int(world)))
        self._graphs.clear()
        self.dp_world = int(world)
        # the gradient bucket moves into the peer-mapped allocation of the library (lcn_dp_bucket): a zero-copy torch
        # view of it through the CUDA array interface replaces the torch-allocated one
        ptr = int(self.lib.lcn_dp_bucket(self.h))

        class _Bucket:
            __cuda_array_interface__ = {"shape": (self.n_params,), "typestr": "<f4", "data": (ptr, False), "version": 2}
        self._dp_bucket_owner = _Bucket()
        self.grads_raw = torch.as_tensor(self._dp_bucket_owner, device=self.device)
        assert self.grads_raw.data_ptr() == ptr

    def dp_enable(self, mode):
        """lcn_dp_enable: 1 / True streamed behind the weight-gradient GEMMs (default), 2 one exchange at the end of the
        backward pass, 0 / False none (backward leaves the local gradient)."""
        L.check(self.lib.lcn_dp_enable(self.h, int(mode)))
        self._graphs.clear()

    def dp_sync_batch_norm(self, on):
        """lcn_dp_sync_batch_norm: True -> every BatchNorm layer of a training step uses the statistics of the global
        batch (all ranks' rows), as one GPU would on the concatenated batch; False (default) -> per-rank statistics.
        Needs a connected engine to turn on."""
        L.check(self.lib.lcn_dp_sync_batch_norm(self.h, int(bool(on))))
        self._graphs.clear()
        self.sync_bn = bool(on)

    # ---- data-parallel exchange: only what backward produces travels (lcn_model_pack_grads) ----
    def pack_grads(self):
        """Gather the nonzero weight blocks + every other tensor of the raw-gradient bucket into self.grads_compact."""
        if getattr(self, "grads_compact", None) is None:
            n = int(self.lib.lcn_model_grad_compact_count(self.h))
            self.grads_compact = torch.empty(n, dtype=torch.float32, device=self.device)
        L.check(self.lib.lcn_model_pack_grads(self.h, _ptr(self.grads_raw), _ptr(self.grads_compact), self._stream()))
        return self.grads_compact

    def unpack_grads(self):
        """Scatter self.grads_compact (all-reduced by the caller) back into the raw-gradient bucket."""
        L.check(self.lib.lcn_model_unpack_grads(self.h, _ptr(self.grads_compact), _ptr(self.grads_raw), self._stream()))
        return self.grads_raw

    def true_grads(self):
        g = torch.empty_like(self.params)
        L.check(self.lib.lcn_model_finalize_grads(self.h, _ptr(self.params), _ptr(self.ws), self.ws.numel(),
                                                  _ptr(self.grads_raw), _ptr(g), self._stream()))
        return g

    def adam(self, beta1=0.9, beta2=0.999, eps=1e-8, dyn=False):
        """TF1 AdamOptimizer.apply_gradients (models_att.py:404-409) + weight re-preparation.
        dyn=True: lr_t is read from self.dyn_dev on the device (CUDA-graph replay); self.step is not advanced."""
        if not dyn:
            self.step += 1
        t = max(self.step, 1)
        lr = self.lr_at(t)
        lr_t = lr * math.sqrt(1.0 - beta2 ** t) / (1.0 - beta1 ** t)
        L.check(self.lib.lcn_model_adam_step(self.h, _ptr(self.params), _ptr(self.adam_m), _ptr(self.adam_v),
                                             _ptr(self.ws), self.ws.numel(), _ptr(self.grads_raw), lr_t, beta1, beta2,
                                             eps, self.regularization, _ptr(self.dyn_dev) if dyn else C.c_void_p(0),
                                             self._stream()))
        self._prepared = True
        return lr

    # ---- CUDA-graph train step ----------------------------------------------------------------
    def _stage_scalars(self, t, beta1=0.9, beta2=0.999):
        """Write lcn_step_scalars{step=t, lr_t} to the device (pinned staging, stream ordered)."""
        lr = self.lr_at(t)
        lr_t = lr * math.sqrt(1.0 - beta2 ** t) / (1.0 - beta1 ** t)
        slot = t % 64
        if self._dyn_ev[slot] is not None:
            self._dyn_ev[slot].synchronize()          # the copy that last used this pinned slot has executed
        buf = self.dyn_pin.numpy()[slot]
        buf[0:8] = np.frombuffer(np.uint64(t).tobytes(), dtype=np.uint8)
        buf[8:12] = np.frombuffer(np.float32(lr_t).tobytes(), dtype=np.uint8)
        self.dyn_dev.copy_(self.dyn_pin[slot], non_blocking=True)
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(self.device))
        self._dyn_ev[slot] = ev
        return lr

    def update_loss_ema(self, decay=0.9):
        """op_loss_average of the reference, run every step (models_att.py:210-212,370-379): EMA of the TOTAL loss
        (mse + regularization * sum l2_loss when regularization != 0) on the device; read it with loss_average()."""
        reg = C.c_void_p(0)
        if self.regularization != 0.0:
            L.check(self.lib.lcn_l2_regularizer(self.h, _ptr(self.params), _ptr(self._reg_scratch), _ptr(self.reg_dev),
                                                self._stream()))
            reg = _ptr(self.reg_dev)
        L.check(self.lib.lcn_loss_ema(_ptr(self.loss_dev), reg, float(self.regularization), float(decay),
                                      _ptr(self.ema_dev), self._stream()))

    def loss_average(self, decay=0.9):
        """averages.average(loss) with TF's zero-debias [TF-sem]: biased / (1 - decay^steps).  One D2H read."""
        biased, steps = self.ema_dev.tolist()
        return biased / (1.0 - decay ** steps) if steps > 0 else 0.0

    def train_step_graph(self, x, labels, dropout=0.0, allreduce=None, packed=False, track_ema=False):
        """train_step() as CUDA-graph replays: the ~60 launches of one step (forward, loss, backward, chain rule,
        Adam, weight re-preparation) are captured once per (batch shape, dropout, buffers) and replayed; the
        per-step scalars (dropout counter, Adam step size) travel through 16 bytes of device memory.
        `x` / `labels` must be the SAME device tensors every call (copy new batches into them).
        allreduce: optional callable run between backward and Adam on the gradient bucket (data parallel);
        then two graphs are replayed around it.  packed=True: the callable receives the packed bucket
        (self.grads_compact: nonzero weight blocks + small tensors); the pack / unpack launches are part of the two
        graphs.  Returns (loss device scalar, learning rate used)."""
        key = (x.data_ptr(), labels.data_ptr(), tuple(x.shape), float(dropout), allreduce is not None, bool(packed),
               bool(track_ema))
        n = x.shape[0]
        if key not in self._graphs:
            self._ensure_ws(n, n, True)
            if not self._prepared:
                self.prepare()
            out = torch.empty((n, J * 3), dtype=torch.float32, device=self.device)
            if packed:
                self.pack_grads()                    # allocates self.grads_compact outside the capture
            self._stage_scalars(self.step + 1)
            # warm-up on a side stream (first-call attribute setup must not happen under capture)
            side = torch.cuda.Stream(device=self.device)
            side.wait_stream(torch.cuda.current_stream(self.device))
            saved = (self.params.clone(), self.adam_m.clone(), self.adam_v.clone(), self.ema_dev.clone())
            with torch.cuda.stream(side):
                self.forward(x, bn_group=n, training=True, dropout=dropout, out=out, dyn=True)
                self.backward(x, labels, dropout)
                if track_ema:
                    self.update_loss_ema()
                self.adam(dyn=True)
            torch.cuda.current_stream(self.device).wait_stream(side)
            self.params.copy_(saved[0]); self.adam_m.copy_(saved[1]); self.adam_v.copy_(saved[2])
            self.ema_dev.copy_(saved[3])
            self.prepare()
            torch.cuda.synchronize(self.device)
            g1 = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g1):
                self.forward(x, bn_group=n, training=True, dropout=dropout, out=out, dyn=True)
                self.backward(x, labels, dropout)
                if track_ema:
                    self.update_loss_ema()           # before Adam: the regulariser is that of the step's parameters
                if allreduce is None:
                    self.adam(dyn=True)
                elif packed:
                    self.pack_grads()
            g2 = None
            if allreduce is not None:
                g2 = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g2):
                    if packed:
                        self.unpack_grads()
                    self.adam(dyn=True)
            self._graphs[key] = (g1, g2, out)
        g1, g2, _ = self._graphs[key]
        lr = self._stage_scalars(self.step + 1)
        g1.replay()
        if g2 is not None:
            allreduce(self.grads_compact if packed else self.grads_raw)
            g2.replay()
        self.step += 1
        self._prepared = True
        self._fwd_geom = (n, n, True)
        return self.loss_dev, lr

    def train_step(self, x, labels, dropout=0.0, out=None, track_ema=False):
        """One sess.run([op_train, op_loss_average]) of the reference (models_att.py:210-212): fwd, loss, bwd, Adam.
        Returns (loss device scalar, learning rate used)."""
        self.forward(x, bn_group=x.shape[0], training=True, dropout=dropout, out=out)
        loss = self.backward(x, labels, dropout)
        if track_ema:
            self.update_loss_ema()
        lr = self.adam()
        return loss, lr

    # ---- optimizer / trainer state (what tf.train.Saver stores next to the variables) ---------------
    def get_state(self):
        """Adam slots, global_step and the loss EMA: with get_params() the complete trainer state."""
        return {"adam_m": self.adam_m.detach().cpu().numpy(), "adam_v": self.adam_v.detach().cpu().numpy(),
                "global_step": np.asarray(self.step, dtype=np.int64), "loss_ema": self.ema_dev.detach().cpu().numpy()}

    def set_state(self, st):
        self.adam_m.copy_(torch.as_tensor(np.asarray(st["adam_m"], dtype=np.float32)))
        self.adam_v.copy_(torch.as_tensor(np.asarray(st["adam_v"], dtype=np.float32)))
        self.step = int(st["global_step"])
        if "loss_ema" in st:
            self.ema_dev.copy_(torch.as_tensor(np.asarray(st["loss_ema"], dtype=np.float32)))

    # ---- the reference's method-level layer API, one kernel launch sequence each ------------------------
    def forward_layers(self, layer_begin, layer_end, n_rows, bn_group=None, x=None, dropout=0.0, out=None):
        """Linear layers [layer_begin, layer_end) with what follows each (BN / LeakyReLU / dropout / residual) on
        the training-layout workspace (lcn_model_forward_layers)."""
        bn_group = n_rows if bn_group is None else int(bn_group)
        size = self._ensure_ws(n_rows, bn_group, True)
        if not self._prepared:
            self.prepare()
        L.check(self.lib.lcn_model_forward_layers(self.h, _ptr(self.params), _ptr(self.ws), size, _ptr(x), n_rows, bn_group,
                                                  float(dropout), self.seed, self.step + 1, int(layer_begin),
                                                  int(layer_end), _ptr(out), self._stream()))
        self._fwd_geom = None

    def write_activation(self, layer, a, bn_group=None):
        """Inject a dense fp32 [n, 17*F] activation as the layer output A_layer (lcn_model_write_tensor)."""
        n = a.shape[0]
        bn_group = n if bn_group is None else int(bn_group)
        size = self._ensure_ws(n, bn_group, True)
        L.check(self.lib.lcn_model_write_tensor(self.h, _ptr(self.ws), size, 1, int(layer), n, bn_group, _ptr(a),
                                                self._stream()))

    def mask_weights(self, w):
        """cgcnn.mask_weights (models_att.py:576-586) on a CUDA float32 [17*Fi, 17*Fo] tensor, current mask values."""
        self.prepare()
        mask = self.read_tensor(3, 0, 128, 128)
        out = torch.empty_like(w)
        L.check(self.lib.lcn_mask_weights(_ptr(w), w.shape[0], w.shape[1], _ptr(mask), _ptr(out), self._stream()))
        return out

    def batch_norm(self, y, bn_name):
        """cgcnn.batch_normalization_warp (models_att.py:588-612) with the gamma / beta of BN layer `bn_name`."""
        g, b = self.tensor(bn_name + "/gamma"), self.tensor(bn_name + "/beta")
        out = torch.empty_like(y)
        L.check(self.lib.lcn_batch_norm(_ptr(y), y.shape[0], y.shape[1] // J, _ptr(g), _ptr(b), 1e-3, _ptr(out),
                                        C.c_void_p(0), self._stream()))
        return out

    def mse_loss(self, pred, labels, with_reg=True):
        """base_model.loss (models_att.py:352-366) on CUDA float32 tensors: mse (+ regularization * sum l2_loss)."""
        out = torch.empty(1, dtype=torch.float32, device=self.device)
        reg = C.c_void_p(0)
        if with_reg and self.regularization != 0.0:
            L.check(self.lib.lcn_l2_regularizer(self.h, _ptr(self.params), _ptr(self._reg_scratch), _ptr(self.reg_dev),
                                                self._stream()))
            reg = _ptr(self.reg_dev)
        L.check(self.lib.lcn_mse_loss(_ptr(pred), _ptr(labels), pred.numel(), reg, float(self.regularization), _ptr(out),
                                      self._stream()))
        return out

    def l2_regularizer(self):
        """tf.add_n(self.regularizers) (models_att.py:364,465-472): sum over w*, b* of sum(v^2)/2, as a float."""
        L.check(self.lib.lcn_l2_regularizer(self.h, _ptr(self.params), _ptr(self._reg_scratch), _ptr(self.reg_dev),
                                            self._stream()))
        return float(self.reg_dev.item())

    def gather_rows(self, src_a, dst_a, idx, src_b=None, dst_b=None):
        """Batch gather of fit (models_att.py:200) from the device-resident set(s): dst[b] = src[idx[b]]."""
        L.check(self.lib.lcn_gather_rows(_ptr(src_a), src_a.shape[1], _ptr(dst_a), _ptr(src_b),
                                         src_b.shape[1] if src_b is not None else 0, _ptr(dst_b), _ptr(idx),
                                         idx.numel(), src_a.shape[0], self._stream()))

    def read_tensor(self, kind, layer, n_rows, bn_group):
        n_groups = (n_rows + bn_group - 1) // bn_group
        P = J * self.F
        if kind in (0, 1, 6):
            shape = (n_groups * bn_group, P)
        elif kind == 2:
            n_lin = 2 + 2 * self.num_layers
            kin = J * (self.in_F if layer == 0 else self.F)
            kout = J * (3 if layer == n_lin - 1 else self.F)
            shape = (kin, kout)
        elif kind == 3:
            shape = (J, J)
        else:
            shape = (n_groups, self.F)
        dst = torch.empty(shape, dtype=torch.float32, device=self.device)
        L.check(self.lib.lcn_model_read_tensor(self.h, _ptr(self.ws), self.ws.numel(), kind, layer, n_rows, bn_group,
                                               _ptr(dst), self._stream()))
        return dst

    def dropout_keep(self, layer, rows, rate, step=None):
        P = J * self.F
        k = torch.empty((rows, P), dtype=torch.uint8, device=self.device)
        L.check(self.lib.lcn_dropout_mask(self.seed, self.step + 1 if step is None else step, layer, rows, P,
                                          float(rate), _ptr(k), self._stream()))
        return k

    # ---- batched predict (base_model.predict, models_att.py:79-132) -------------------------------
    def predict(self, data, batch_size, chunk_groups=None, out=None):
        """data: [N, 17*in_F] array (host).  Batches of `batch_size` poses are BN groups; the last one is
        zero padded (the zero rows take part in the statistics) exactly like the reference.  Returns
        float64 [N, 51].

        Pipelined: chunks of `chunk_groups` batches rotate through two pinned input / output buffers and two device
        buffer pairs; the H2D copy of chunk i+1 (copy stream) and the D2H copy of chunk i-1 (drain stream) overlap the
        forward pass of chunk i, and the host only ever waits for the chunk before the previous one."""
        data = np.ascontiguousarray(data, dtype=np.float32)
        n = data.shape[0]
        if chunk_groups is None:
            chunk_groups = max(1, 32768 // batch_size)
        chunk = min(chunk_groups * batch_size, max(n, 1))
        preds = np.empty((n, J * 3), dtype=np.float64) if out is None else out
        if n == 0:
            return preds
        self._ensure_ws(chunk, batch_size, False)
        if not self._prepared:
            self.prepare()
        dev = self.device
        main = torch.cuda.current_stream(dev)
        if getattr(self, "_pp", None) is None or self._pp["chunk"] < chunk or self._pp["cols"] != data.shape[1]:
            self._pp = {"chunk": chunk, "cols": data.shape[1],
                        "pin_in": [torch.empty((chunk, data.shape[1]), dtype=torch.float32).pin_memory() for _ in range(2)],
                        "pin_out": [torch.empty((chunk, J * 3), dtype=torch.float32).pin_memory() for _ in range(2)],
                        "x": [torch.empty((chunk, data.shape[1]), dtype=torch.float32, device=dev) for _ in range(2)],
                        "o": [torch.empty((chunk, J * 3), dtype=torch.float32, device=dev) for _ in range(2)],
                        "copy_s": torch.cuda.Stream(device=dev), "drain_s": torch.cuda.Stream(device=dev)}
        pp = self._pp
        copy_s, drain_s = pp["copy_s"], pp["drain_s"]
        copied = [torch.cuda.Event(), torch.cuda.Event()]
        computed = [torch.cuda.Event(), torch.cuda.Event()]
        drained, drain_ev = [None, None], [None, None]
        spans = [None, None]
        copy_s.wait_stream(main)
        drain_s.wait_stream(main)

        def finish(b):
            if drained[b] is not None:
                drained[b].synchronize()
                lo, hi = spans[b]
                preds[lo:hi] = pp["pin_out"][b][: hi - lo].numpy()
                drained[b] = None

        for i, lo in enumerate(range(0, n, chunk)):
            hi = min(lo + chunk, n)
            b = i & 1
            finish(b)                                   # chunk i-2: its pinned buffers are free again
            pp["pin_in"][b][: hi - lo].copy_(torch.from_numpy(data[lo:hi]))
            with torch.cuda.stream(copy_s):
                if i >= 2:
                    copy_s.wait_event(computed[b])      # the forward pass that read x[b] has finished
                pp["x"][b][: hi - lo].copy_(pp["pin_in"][b][: hi - lo], non_blocking=True)
                copied[b].record(copy_s)
            main.wait_event(copied[b])
            if i >= 2:
                main.wait_event(drain_ev[b])            # the D2H copy that read o[b] has finished
            self.forward(pp["x"][b][: hi - lo], bn_group=batch_size, training=False, out=pp["o"][b][: hi - lo])
            computed[b].record(main)
            with torch.cuda.stream(drain_s):
                drain_s.wait_event(computed[b])
                pp["pin_out"][b][: hi - lo].copy_(pp["o"][b][: hi - lo], non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(drain_s)
            drained[b] = drain_ev[b] = ev
            spans[b] = (lo, hi)
        finish(0)
        finish(1)
        main.wait_stream(copy_s)
        main.wait_stream(drain_s)
        return preds


def eval_mpjpe(pred, gt, box=None, cam=None, root_depth=None, protocol2=False, action=None, n_actions=0,
               want_err=True, want_pose=False, camera_frame=False):
    """Batched evaluate.py:53-61.  CUDA float32 tensors: pred/gt [n,17,3], box [n,4], cam [n,4]=(fx,fy,cx,cy),
    root_depth [n]; action int32 [n] or None.  camera_frame=True: pred is already in the camera frame.
    Returns (err [n,17] or None, sums float64 [n_actions+1, 19]) and the transformed poses when want_pose."""
    lib = L.load()
    n = pred.shape[0]
    dev = pred.device
    for t in (pred, gt, box, cam, root_depth):
        assert t is None or (t.is_cuda and t.dtype == torch.float32 and t.is_contiguous())
    err = torch.empty((n, J), dtype=torch.float32, device=dev) if want_err else None
    pose = torch.empty((n, J, 3), dtype=torch.float32, device=dev) if want_pose else None
    na = int(n_actions) if action is not None else 0
    sums = torch.zeros((na + 1, 19), dtype=torch.float64, device=dev)
    flags = (L.LCN_EVAL_PROTOCOL2 if protocol2 else 0) | (L.LCN_EVAL_CAMERA_FRAME if camera_frame else 0)
    L.check(lib.lcn_eval_mpjpe(_ptr(pred), _ptr(gt), _ptr(box), _ptr(cam), _ptr(root_depth), _ptr(action), na, n,
                               flags, _ptr(err), _ptr(pose), _ptr(sums),
                               C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
    if want_pose:
        return err, sums, pose
    return err, sums
