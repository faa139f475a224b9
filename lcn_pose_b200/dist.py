"""Host-side multi-GPU plumbing (SURVEY 8(e)): one process per GPU, torch.distributed for the rendezvous.

* Inference / evaluation shard the pose set at BatchNorm-group granularity (the reference's BN uses batch statistics at
  inference too, models_att.py:588-612 + SURVEY 9-Q2, so a batch of `batch_size` consecutive poses is the unit of
  independence): no collective on the data path, one small all-reduce of the per-joint error sums at the end.
* Data-parallel training all-reduces ONE bucket (the raw gradients, packed to the nonzero weight blocks + the small
  tensors: average_gradients_packed; or the flat parameter-layout vector: average_gradient_bucket) between backward
  and the fused Adam step.  BatchNorm statistics have two semantics:
  - sync_bn=False (default): per GPU -- every rank normalises over its own rows, i.e. the reference trained at the
    per-GPU batch;
  - sync_bn=True (lcn_dp_sync_batch_norm): over the global batch -- the forward pass equals one GPU's on the
    concatenated batch, and the exchanged gradient is that of the mean of the ranks' losses (for equal shards, the
    single-GPU gradient on the concatenated batch).  The moments travel over NVLink peer memory, one flag round trip
    per BatchNorm layer in the forward and in the backward pass, so it needs init_native_dp even in the "packed" mode.
* Two exchange modes for training.  "p2p" (default, init_native_dp + LcnEngine.train_step_graph): lcn_model_backward ends
  with the library's own two-shot all-reduce of the packed bucket over NVLink peer memory (csrc/lcn_dp.cu); the whole
  step is ONE CUDA graph.  "packed": the round-1 path -- backward, pack the nonzero blocks, one torch.distributed (NCCL)
  all-reduce, unpack, Adam -- two graphs around the library collective; kept as the reference point.
Everything else here is backend agnostic (nccl on GPUs, gloo in the CPU tests)."""
import torch
import torch.distributed as dist


def shard_groups(n_rows, batch_size, rank, world):
    """Contiguous range of BN groups of this rank -> (row_begin, row_end).  Groups are ceil(n_rows / batch_size)
    batches as base_model.predict forms them (models_att.py:86-97); the last one may be partial (zero padded by
    the kernels).  Ranks get floor/ceil(groups / world) groups, earlier ranks the larger share."""
    groups = (n_rows + batch_size - 1) // batch_size
    base, extra = divmod(groups, world)
    g0 = rank * base + min(rank, extra)
    g1 = g0 + base + (1 if rank < extra else 0)
    return min(g0 * batch_size, n_rows), min(g1 * batch_size, n_rows)


def all_reduce_eval_sums(sums, group=None):
    """Sum the evaluator's accumulators ([n_actions+1, 19] float64: 17 per-joint error sums, count, PCK hits) over
    the ranks; the MPJPE means are then sums[:, :17].sum() / (17 * count) on every rank."""
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(sums, op=dist.ReduceOp.SUM, group=group)
    return sums


def average_gradient_bucket(bucket, group=None):
    """Data-parallel exchange step: mean of the flat raw-gradient bucket over the ranks (one collective)."""
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        if dist.get_backend(group) == "nccl":
            dist.all_reduce(bucket, op=dist.ReduceOp.AVG, group=group)      # averaged inside the collective
        else:
            dist.all_reduce(bucket, op=dist.ReduceOp.SUM, group=group)
            bucket.div_(dist.get_world_size(group))
    return bucket


def average_gradients_packed(engine, group=None):
    """The same exchange on the packed bucket: LcnEngine.pack_grads() leaves out the never-written entries of the
    masked-out joint-pair blocks (40 % of the parameter-layout bucket for knn=3), one collective, unpack.  No-op (and no
    pack / unpack launches) in a single process."""
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        average_gradient_bucket(engine.pack_grads(), group)
        engine.unpack_grads()
    return engine.grads_raw


def broadcast_parameters(flat_params, src=0, group=None):
    """Replicas start from rank `src`'s parameters (the reference has a single process)."""
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.broadcast(flat_params, src=src, group=group)
    return flat_params


def init_native_dp(engine, group=None, sync_bn=False):
    """Connect the engine's exchange buffers across the ranks (lcn_dp_export / lcn_dp_connect): every rank exports the CUDA
    IPC handle of its buffer, torch.distributed all-gathers them (any backend).  Collective over `group`.  sync_bn=True
    also turns on BatchNorm statistics of the global batch (LcnEngine.dp_sync_batch_norm).  No-op in a single process."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return False
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    handles = [None] * world
    dist.all_gather_object(handles, engine.dp_export(world), group=group)
    engine.dp_connect(handles, rank, world)
    if sync_bn:
        engine.dp_sync_batch_norm(True)
    dist.barrier(group)                    # nobody starts exchanging before everybody has mapped everybody
    return True


def dp_train_step(engine, x, labels, dropout=0.0, mode="p2p", group=None, graph=True, sync_bn=False):
    """One data-parallel train step on this rank's shard of the global batch; returns (loss, lr) like train_step.
    mode "p2p": exchange inside lcn_model_backward, streamed behind the weight-gradient GEMMs (init_native_dp is run on
    first use); "p2p-end": the same kernels, one exchange at the end of the backward pass; "packed": torch all-reduce of
    the packed bucket between backward and Adam.  sync_bn=True: BatchNorm over the global batch (module docstring); the
    "packed" mode then connects the engine as well and turns off only the exchange inside backward."""
    multi = dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1
    if multi and getattr(engine, "dp_world", 1) == 1 and (mode in ("p2p", "p2p-end") or (mode == "packed" and sync_bn)):
        init_native_dp(engine, group, sync_bn)
        if mode != "packed":
            engine.dp_enable(1 if mode == "p2p" else 2)
    if multi and abs(getattr(engine, "dp_world", 1)) > 1 and getattr(engine, "sync_bn", False) != bool(sync_bn):
        engine.dp_sync_batch_norm(sync_bn)
    if mode in ("p2p", "p2p-end"):
        return engine.train_step_graph(x, labels, dropout) if graph else engine.train_step(x, labels, dropout)
    if mode != "packed":
        raise ValueError("mode must be 'p2p', 'p2p-end' or 'packed'")
    if getattr(engine, "dp_world", 1) > 1:
        engine.dp_enable(False)          # the torch-level exchange below replaces the one inside backward
        engine.dp_world = -engine.dp_world
    if not multi:
        return engine.train_step_graph(x, labels, dropout) if graph else engine.train_step(x, labels, dropout)
    if graph:
        return engine.train_step_graph(x, labels, dropout, lambda b: average_gradient_bucket(b, group), packed=True)
    engine.forward(x, bn_group=x.shape[0], training=True, dropout=dropout)
    loss = engine.backward(x, labels, dropout)
    average_gradient_bucket(engine.pack_grads(), group)
    engine.unpack_grads()
    return loss, engine.adam()
