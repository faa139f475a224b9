"""Float64 specification of synchronised BatchNorm under data parallelism (lcn_dp_sync_batch_norm), built from the
oracle's pieces (oracle/lcn_oracle.py).  W ranks hold shards x_0 .. x_{W-1}; every BatchNorm layer of the forward pass
uses the mean / biased variance over ALL rows x 17 joints; rank r's backward pass starts from d_r = dL_r/dout (L_r its
local MSE) and applies dz = gamma rstd (d - S1/N - xhat S2/N) with S1, S2 summed over every rank's rows and N = 17 x
global rows.  Each rank's gradient is then W times its share of the gradient of (1/W) sum_r L_r, and the mean over the
ranks (what the bucket exchange computes) is that gradient.  gamma / beta gradients are per-rank sums, averaged the same
way.  The device kernels implement exactly this; tests/test_sync_bn_oracle.py pins it against single-batch references."""
import numpy as np

from oracle import lcn_oracle as O

J = O.J


def loss_and_grads_sharded(cfg, p, shards, labels, keep_masks=None, dropout_rate=0.0):
    """shards / labels: lists of W arrays [n_r, 17*in_F] / [n_r, 51]; keep_masks: per shard, a list of 1+2L keep arrays
    [n_r, 17*F] (or None).  Returns (mean of the per-shard losses, mean of the per-shard gradients, per-shard
    gradients)."""
    W = len(shards)
    xs = [np.asarray(x, dtype=np.float64) for x in shards]
    ys = [np.asarray(y, dtype=np.float64) for y in labels]
    ns = [x.shape[0] for x in xs]
    N = float(sum(ns) * J)
    F = cfg.F
    mask = O.mask_values(cfg, p)
    wn, bn_, bnn = O.weight_names(cfg), O.bias_names(cfg), O.bn_names(cfg)
    scale = 1.0 / (1.0 - dropout_rate) if dropout_rate > 0 else 1.0
    caches = [[] for _ in range(W)]

    def layer_fwd(a_in, l, with_bn_act):
        w = p[wn[l]].astype(np.float64)
        wm, wc, norm = O.effective_weight(cfg, w, mask)
        zs = [a @ wm + p[bn_[l]].astype(np.float64) for a in a_in]
        recs = [{"a_in": a, "wm": wm, "wc": wc, "norm": norm, "z": z} for a, z in zip(a_in, zs)]
        ys_ = zs
        if with_bn_act:
            if cfg.batch_norm:
                g = p[bnn[l] + "/gamma"].astype(np.float64)
                b = p[bnn[l] + "/beta"].astype(np.float64)
                z3 = [z.reshape(-1, J, F) for z in zs]
                mu = sum(z.sum(axis=(0, 1)) for z in z3) / N                     # pooled moments
                var = sum(((z - mu) ** 2).sum(axis=(0, 1)) for z in z3) / N
                rstd = 1.0 / np.sqrt(var + O.BN_EPS)
                ys_ = []
                for r, z in enumerate(z3):
                    xhat = (z - mu) * rstd
                    recs[r].update(xhat=xhat.reshape(-1, J * F), mu=mu, rstd=rstd)
                    ys_.append((g * xhat + b).reshape(-1, J * F))
            out = []
            for r, y in enumerate(ys_):
                recs[r]["ybn"] = y
                y = np.where(y > 0, y, O.LRELU_ALPHA * y)
                if dropout_rate > 0:
                    recs[r]["keep"] = keep_masks[r][l]
                    y = y * keep_masks[r][l] * scale
                out.append(y)
            ys_ = out
        for r in range(W):
            recs[r]["out"] = ys_[r]
            caches[r].append(recs[r])
        return ys_

    y = layer_fwd(xs, 0, True)
    l = 1
    for _ in range(cfg.num_layers):
        xin = y
        y = layer_fwd(layer_fwd(xin, l, True), l + 1, True)
        if cfg.residual:
            y = [a + b for a, b in zip(xin, y)]
        l += 2
    y = layer_fwd(y, l, False)
    outs = []
    for r in range(W):
        y3 = y[r].reshape(-1, J, 3).copy()
        y3[:, :, :2] += xs[r].reshape(-1, J, cfg.in_F)[:, :, :2]
        outs.append(y3.reshape(-1, J * 3))

    grads = [{} for _ in range(W)]
    dmask = [np.zeros((J, J)) for _ in range(W)]

    def layer_bwd(l, d_out, with_bn_act):
        ds = list(d_out)
        if with_bn_act:
            for r in range(W):
                rec = caches[r][l]
                if dropout_rate > 0:
                    ds[r] = ds[r] * rec["keep"] * scale
                ds[r] = ds[r] * np.where(rec["ybn"] > 0, 1.0, O.LRELU_ALPHA)
            if cfg.batch_norm:
                gam = p[bnn[l] + "/gamma"].astype(np.float64)
                d3 = [d.reshape(-1, J, F) for d in ds]
                xh3 = [caches[r][l]["xhat"].reshape(-1, J, F) for r in range(W)]
                s1 = [d.sum(axis=(0, 1)) for d in d3]                             # local sums: dbeta, dgamma
                s2 = [(d * x).sum(axis=(0, 1)) for d, x in zip(d3, xh3)]
                S1, S2 = sum(s1), sum(s2)                                         # exchanged
                for r in range(W):
                    grads[r][bnn[l] + "/gamma"] = s2[r]
                    grads[r][bnn[l] + "/beta"] = s1[r]
                    ds[r] = (gam * caches[r][l]["rstd"] * (d3[r] - S1 / N - xh3[r] * S2 / N)).reshape(-1, J * F)
        d_in = []
        fi, fo = cfg.layer_dims(l)
        for r in range(W):
            rec = caches[r][l]
            dz = ds[r]
            grads[r][bn_[l]] = dz.sum(axis=0)
            dwm = rec["a_in"].T @ dz
            d_in.append(dz @ rec["wm"].T)
            dwm4 = dwm.reshape(J, fi, J, fo)
            dmask[r] += (dwm4 * rec["wc"].reshape(J, fi, J, fo)).sum(axis=(1, 3))
            dwc = (dwm4 * mask.reshape(J, 1, J, 1)).reshape(J * fi, J * fo)
            w = p[wn[l]].astype(np.float64)
            if cfg.max_norm and rec["norm"] > 1.0:
                nrm = rec["norm"]
                grads[r][wn[l]] = dwc / nrm - w * ((dwc * w).sum() / nrm ** 3)
            else:
                grads[r][wn[l]] = dwc
        return d_in

    d = [2.0 * (o - t) / (o.shape[0] * J * 3) for o, t in zip(outs, ys)]           # d L_r / d out_r
    last = cfg.n_lin - 1
    d = layer_bwd(last, d, False)
    l = last - 1
    for _ in range(cfg.num_layers):
        d_block_out = d
        d = layer_bwd(l - 1, layer_bwd(l, d_block_out, True), True)
        if cfg.residual:
            d = [a + b for a, b in zip(d, d_block_out)]
        l -= 2
    layer_bwd(0, d, True)

    if cfg.trainable_mask():
        sup = (cfg.neighbour_matrix.T != 0)
        var = p["mask"].astype(np.float64)
        e = np.exp(var - var.max(axis=0, keepdims=True))
        soft = e / e.sum(axis=0, keepdims=True)
        for r in range(W):
            dsoft = dmask[r] * sup
            grads[r]["mask"] = soft * (dsoft - (soft * dsoft).sum(axis=0, keepdims=True))
    if cfg.regularization is not None and cfg.regularization != 0:
        for r in range(W):
            for n in O.weight_names(cfg) + O.bias_names(cfg):
                grads[r][n] = grads[r][n] + cfg.regularization * p[n].astype(np.float64)
    losses = [O.mse_loss(o, t) + O.reg_loss(cfg, p) for o, t in zip(outs, ys)]
    mean = {k: sum(g[k] for g in grads) / W for k in grads[0]}
    return float(np.mean(losses)), mean, grads


def torch_reference(cfg, p, shards, labels, keep_masks=None, dropout_rate=0.0):
    """The same objective by torch autograd on the concatenated batch (pooled BatchNorm by construction):
    (1/W) sum_r MSE(out[rows of r], labels_r).  Returns (loss, grads)."""
    import torch
    from oracle import torch_restatement as R
    tp = R.build_params(p)
    x = torch.tensor(np.concatenate(shards), dtype=torch.float64)
    km = None
    if dropout_rate > 0:
        km = [torch.tensor(np.concatenate([k[l] for k in keep_masks]), dtype=torch.float64)
              for l in range(len(keep_masks[0]))]
    out = R.forward(cfg, tp, x, dropout_rate, km)
    loss, r0 = 0.0, 0
    for y in labels:
        n = y.shape[0]
        loss = loss + ((out[r0:r0 + n] - torch.tensor(y, dtype=torch.float64)) ** 2).mean()
        r0 += n
    loss = loss / len(labels)
    loss.backward()
    return float(loss.detach()), {k: v.grad.numpy() for k, v in tp.items() if v.grad is not None}
