"""Training step of the sem-seg networks on the GPU (SURVEY.md section 8f rank 3).

Reference: PointNet/train_semseg.py:164-179 -- ``classifier.train()``; ``seg_pred, trans_feat = classifier(points)``;
``loss = criterion(seg_pred, target, trans_feat, weights)`` (weighted NLL, models/pointnet2_sem_seg.py:43-49);
``loss.backward()``; ``optimizer.step()`` with the Adam of :125-132 -- over the modules of
PointNet/models/pointnet_util.py in train mode (BatchNorm on batch statistics with running-stat updates,
``Dropout(0.5)`` active in the head, pointnet2_sem_seg.py:18,35).

The attack path's kernels are reused as they are (FPS, ball query, 3-NN, grouping gather, shared-MLP GEMMs and their
dgrad, neighbourhood max-pool, interpolation, deterministic segmented sums); csrc/train.cu adds batch statistics and their
backward, weight / bias gradients (split-K, ordered), the weighted NLL and Adam.  Two ways in:

* the reference's own loop works unchanged: ``model.train()(x)`` returns ``(logp, l4_points)`` through an autograd
  function whose backward fills ``.grad`` of every parameter, so ``criterion`` / ``loss.backward()`` /
  ``torch.optim.Adam.step()`` run as in train_semseg.py;
* ``Trainer`` does the same step without autograd in between: parameters flattened into one buffer, loss and its
  gradient from ``psg_nll_loss``, one fused Adam kernel.

No CPU fallback: CUDA tensors only.  FPS starts are drawn on the CPU generator per set-abstraction level exactly as the
reference does (pointnet_util.py:75); the dropout keep-mask comes from the device generator (``bernoulli_``) as
``nn.Dropout`` on a CUDA tensor does, or is passed in (parity tests inject the oracle's mask).
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional

import torch

from . import _lib as L
from .engine import MLP_FP32
from .tlayout import TTensor

_GRID_MIN_N = 1024


def _stream():
    return torch.cuda.current_stream().cuda_stream


class _Layer:
    """One 1x1 conv (+ BatchNorm + ReLU) of the network with its device-resident operand packing."""

    def __init__(self, conv, bn, perm=None):
        self.conv, self.bn = conv, bn
        w = conv.weight
        self.cout, self.cin = w.shape[0], w.shape[1]
        self.perm = perm            # input-column permutation (SSG first SA layer: reference order xyz | feats)
        self.h = L.psg_mlp_create_device(self.cin, self.cout)
        if not self.h:
            raise L.PsgError("psg_mlp_create_device failed")

    def load(self):
        w = self.conv.weight.detach().reshape(self.cout, self.cin)
        if self.perm is not None:
            w = w[:, self.perm]
        w = w.contiguous()
        self._w_keep = w
        L.psg_mlp_load(self.h, w.data_ptr(), self.conv.bias.detach().data_ptr(), _stream())

    def __del__(self):
        h, self.h = getattr(self, "h", None), None
        destroy = getattr(L, "psg_mlp_destroy", None)
        if h and destroy is not None:
            destroy(h)


def _tt(rows, channels, dev):
    """T-layout buffer; padded columns zeroed when the width is not a multiple of 16 (they feed GEMMs)."""
    return TTensor(rows, channels, dev, zero=(channels % 16 != 0))


class TrainEngine:
    """Train-mode forward and full backward (parameter gradients) of one sem-seg model."""

    def __init__(self, model, mlp_mode: int = MLP_FP32):
        self.model = model
        self.mode = mlp_mode
        self.dev = next(model.parameters()).device
        if self.dev.type != "cuda":
            raise RuntimeError("pointsecguard_b200 training runs on CUDA devices only (no CPU fallback)")
        self.msg = hasattr(model.sa1, "conv_blocks")
        with torch.cuda.device(self.dev):
            self.sa = []
            for sa in (model.sa1, model.sa2, model.sa3, model.sa4):
                if self.msg:
                    branches = []
                    for i, (r, k) in enumerate(zip(sa.radius_list, sa.nsample_list)):
                        branches.append((float(r), int(k), [_Layer(c, b) for c, b in zip(sa.conv_blocks[i], sa.bn_blocks[i])]))
                else:
                    layers = []
                    for j, (c, b) in enumerate(zip(sa.mlp_convs, sa.mlp_bns)):
                        cin = c.weight.shape[1]
                        perm = list(range(3, cin)) + [0, 1, 2] if j == 0 else None
                        layers.append(_Layer(c, b, perm))
                    branches = [(float(sa.radius), int(sa.nsample), layers)]
                self.sa.append((int(sa.npoint), branches))
            self.fp = [[_Layer(c, b) for c, b in zip(fp.mlp_convs, fp.mlp_bns)]
                       for fp in (model.fp1, model.fp2, model.fp3, model.fp4)]          # fine -> coarse
            self.conv1 = _Layer(model.conv1, model.bn1)
            self.conv2 = _Layer(model.conv2, None)
        self.ncls = model.conv2.out_channels
        self._bn_ws = None
        self._wg_ws = None
        self.ctx = None

    # ---- helpers ----------------------------------------------------------------------------------
    def layers(self) -> List[_Layer]:
        out = []
        for _, branches in self.sa:
            for _, _, ls in branches:
                out += ls
        for ls in self.fp:
            out += ls
        return out + [self.conv1, self.conv2]

    def _bn_workspace(self, C_):
        need = L.psg_bn_workspace(C_)
        if self._bn_ws is None or self._bn_ws.numel() < need:
            self._bn_ws = torch.empty(need, dtype=torch.uint8, device=self.dev)
        return self._bn_ws

    def _wg_workspace(self, cout, cin, rows):
        need = L.psg_wgrad_workspace(cout, cin, rows)
        if self._wg_ws is None or self._wg_ws.numel() < need:
            self._wg_ws = torch.empty(need, dtype=torch.uint8, device=self.dev)
        return self._wg_ws

    def _conv_bn_relu(self, layer: _Layer, a1, k1, a2, k2, rows):
        """z = conv(x); y = relu(bn_train(z)).  Returns the record the backward needs."""
        st = _stream()
        z = _tt(rows, layer.cout, self.dev)
        L.psg_mlp_forward(layer.h, a1.ptr, a1.wchunks, 0, k1, a2.ptr if a2 is not None else None,
                          a2.wchunks if a2 is not None else 0, 0, k2, rows, z.ptr, z.wchunks, 0, self.mode, st)
        rec = {"layer": layer, "a1": a1, "k1": k1, "a2": a2, "k2": k2, "z": z, "rows": rows}
        bn = layer.bn
        if bn is None:
            rec["y"] = z
            return rec
        y = _tt(rows, layer.cout, self.dev)
        mean = torch.empty(layer.cout, dtype=torch.float32, device=self.dev)
        invstd = torch.empty_like(mean)
        ws = self._bn_workspace(layer.cout)
        track = bn.track_running_stats and bn.running_mean is not None
        if track:
            bn.num_batches_tracked += 1
        # nn.BatchNorm: momentum None is the cumulative average, factor 1 / num_batches_tracked counted after this batch
        mom = float(bn.momentum) if bn.momentum is not None else (1.0 / float(bn.num_batches_tracked) if track else 0.0)
        L.psg_bn_train_forward(z.ptr, z.wchunks, rows, layer.cout, bn.weight.data_ptr(), bn.bias.data_ptr(),
                               bn.running_mean.data_ptr() if track else None, bn.running_var.data_ptr() if track else None,
                               mom, float(bn.eps), y.ptr, y.wchunks, 1, mean.data_ptr(), invstd.data_ptr(), ws.data_ptr(),
                               ws.numel(), st)
        rec.update(y=y, mean=mean, invstd=invstd)
        return rec

    def _chain_backward(self, recs, dy, grads, need_input_grad=True):
        """dy: gradient w.r.t. the (post-ReLU) output of the last layer of ``recs`` -> gradient w.r.t. the chain input
        (T-layout, width = padded input width of the first layer) or None."""
        st = _stream()
        cur = dy
        for j in range(len(recs) - 1, -1, -1):
            r = recs[j]
            layer, rows = r["layer"], r["rows"]
            bn = layer.bn
            if bn is not None:
                dg = torch.empty(layer.cout, dtype=torch.float32, device=self.dev)
                db_ = torch.empty_like(dg)
                ws = self._bn_workspace(layer.cout)
                L.psg_bn_train_backward(cur.ptr, cur.wchunks, r["y"].ptr, r["y"].wchunks, r["z"].ptr, r["z"].wchunks, rows,
                                        layer.cout, bn.weight.data_ptr(), r["mean"].data_ptr(), r["invstd"].data_ptr(),
                                        dg.data_ptr(), db_.data_ptr(), cur.ptr, cur.wchunks, ws.data_ptr(), ws.numel(), st)
                grads[bn.weight] = dg
                grads[bn.bias] = db_
            # weight / bias gradient
            k1c, k2c = r["k1"] * 4, r["k2"] * 4
            if r["a2"] is None:
                k1c = layer.cin                      # single source: exact input width (padding columns are zero)
            dW = torch.empty(layer.cout, layer.cin, dtype=torch.float32, device=self.dev)
            dB = torch.empty(layer.cout, dtype=torch.float32, device=self.dev)
            ws = self._wg_workspace(layer.cout, layer.cin, rows)
            L.psg_conv_wgrad(cur.ptr, cur.wchunks, layer.cout, r["a1"].ptr, r["a1"].wchunks, 0, k1c,
                             r["a2"].ptr if r["a2"] is not None else None, r["a2"].wchunks if r["a2"] is not None else 0, 0,
                             k2c if r["a2"] is not None else 0, rows, dW.data_ptr(), dB.data_ptr(), 0, ws.data_ptr(), ws.numel(), st)
            if layer.perm is not None:
                full = torch.empty_like(dW)
                full[:, layer.perm] = dW
                dW = full
            grads[layer.conv.weight] = dW.view_as(layer.conv.weight)
            grads[layer.conv.bias] = dB
            if j == 0 and not need_input_grad:
                return None
            kpad = (layer.cin + 15) // 16 * 16
            dx = TTensor(rows, kpad, self.dev)
            L.psg_mlp_backward(layer.h, cur.ptr, cur.wchunks, rows, dx.ptr, dx.wchunks, None, 0, self.mode, st)
            cur = dx
        return cur

    # ---- forward ----------------------------------------------------------------------------------
    def forward(self, x: torch.Tensor, dropout_mask: Optional[torch.Tensor] = None, starts=None):
        """x [B,9,N] float32 CUDA -> (logp [B,N,ncls], l4_points [B,C4,16]).  ``dropout_mask`` [B,128,N] of 0/1 keeps
        (None: drawn on the device generator); ``starts``: optional list of four int64 [B] CPU tensors (FPS starts)."""
        if not x.is_cuda or x.dtype != torch.float32 or x.dim() != 3 or x.shape[1] != 9:
            raise ValueError("expected a float32 CUDA tensor [B, 9, N]")
        dev, st = self.dev, _stream()
        B, _, N = x.shape
        for l in self.layers():
            l.load()
        feats0, xyz0 = TTensor.from_channels_first(x.detach(), want_xyz=True)
        feats, xyzs, widths = [feats0], [xyz0], [9]
        sa_recs = []
        for li, (S, branches) in enumerate(self.sa):
            R = xyzs[-1].shape[1]
            start = starts[li] if starts is not None else torch.randint(0, R, (B,), dtype=torch.long)     # pointnet_util.py:75
            start_d = start.to(device=dev, dtype=torch.int32)
            fps_idx = torch.empty(B, S, dtype=torch.int32, device=dev)
            new_xyz = torch.empty(B, S, 3, dtype=torch.float32, device=dev)
            wsb = L.psg_fps_workspace(B, R)
            ws = torch.empty(max(wsb, 16), dtype=torch.uint8, device=dev)
            L.psg_fps(xyzs[-1].data_ptr(), B, B, R, S, start_d.data_ptr(), fps_idx.data_ptr(), new_xyz.data_ptr(), ws.data_ptr(),
                      wsb, st)
            ctot = sum(ls[-1].cout for _, _, ls in branches)
            out = _tt(B * S, ctot, dev)
            D = widths[-1]
            level = []
            col = 0
            for radius, K, ls in branches:
                idx = torch.empty(B, S, K, dtype=torch.int32, device=dev)
                rr, kk = (C.c_double * 1)(radius), (C.c_int * 1)(K)
                if R >= _GRID_MIN_N:
                    gb = L.psg_ball_grid_workspace(B, R)
                    gws = torch.empty(gb, dtype=torch.uint8, device=dev)
                    L.psg_ball_query_grid(xyzs[-1].data_ptr(), B, B, R, new_xyz.data_ptr(), S, 1, rr, kk, idx.data_ptr(), None,
                                          gws.data_ptr(), gb, st)
                else:
                    L.psg_ball_query(xyzs[-1].data_ptr(), B, B, R, new_xyz.data_ptr(), S, 1, rr, kk, idx.data_ptr(), None, st)
                rows = B * S * K
                G = TTensor(rows, D + 3, dev)
                L.psg_group_points(feats[-1].ptr, feats[-1].wchunks, D, xyzs[-1].data_ptr(), B, R, new_xyz.data_ptr(),
                                   idx.data_ptr(), B, S, K, G.ptr, G.cpad, st)
                recs, cur, k = [], G, G.wchunks
                for layer in ls:
                    rec = self._conv_bn_relu(layer, cur, k, None, 0, rows)
                    recs.append(rec)
                    cur, k = rec["y"], rec["y"].wchunks
                arg = torch.empty(B * S * cur.cpad, dtype=torch.uint8, device=dev)
                L.psg_group_max(cur.ptr, cur.wchunks, B * S, K, cur.cpad, out.ptr, out.wchunks, col // 4, arg.data_ptr(), st)
                level.append({"idx": idx, "recs": recs, "arg": arg, "col": col, "K": K, "cw": cur.cpad})
                col += ls[-1].cout
            sa_recs.append({"branches": level, "out": out, "S": S, "R": R, "D": D})
            feats.append(out)
            xyzs.append(new_xyz)
            widths.append(ctot)
        # feature propagation, coarse to fine: fp4 (fine level 3) ... fp1 (fine level 0)
        up, upw = feats[4], widths[4]
        fp_recs = [None] * 4
        for f in (3, 2, 1, 0):
            Nf, Nc = xyzs[f].shape[1], xyzs[f + 1].shape[1]
            rows = B * Nf
            nn_idx = torch.empty(B, Nf, 3, dtype=torch.int32, device=dev)
            nn_w = torch.empty(B, Nf, 3, dtype=torch.float32, device=dev)
            L.psg_three_nn(xyzs[f].data_ptr(), B, B, Nf, xyzs[f + 1].data_ptr(), Nc, nn_idx.data_ptr(), nn_w.data_ptr(), None, st)
            interp = _tt(rows, upw, dev)
            L.psg_interpolate(up.ptr, up.wchunks, Nc, nn_idx.data_ptr(), nn_w.data_ptr(), B, Nf, up.cpad, interp.ptr,
                              interp.wchunks, 0, st)
            if f > 0:
                a1, k1, a2, k2 = feats[f], feats[f].wchunks, interp, interp.wchunks
                if widths[f] % 16 or upw % 16:
                    raise L.PsgError("feature propagation: level widths must be multiples of 16")
            else:
                a1, k1, a2, k2 = interp, interp.wchunks, None, 0
            recs = []
            for layer in self.fp[f]:
                rec = self._conv_bn_relu(layer, a1, k1, a2, k2, rows)
                recs.append(rec)
                a1, k1, a2, k2 = rec["y"], rec["y"].wchunks, None, 0
            fp_recs[f] = {"recs": recs, "nn_idx": nn_idx, "nn_w": nn_w, "Nf": Nf, "Nc": Nc, "C1": widths[f] if f > 0 else 0, "C2": upw}
            up, upw = recs[-1]["y"], self.fp[f][-1].cout
        rows0 = B * N
        r1 = self._conv_bn_relu(self.conv1, up, up.wchunks, None, 0, rows0)
        h = r1["y"]
        # Dropout(0.5): keep-mask * 2 (pointnet2_sem_seg.py:18,35)
        if dropout_mask is None:
            dropout_mask = torch.empty(B, self.conv1.cout, N, dtype=torch.float32, device=dev).bernoulli_(0.5)
        mk = TTensor.from_channels_first(dropout_mask.to(device=dev, dtype=torch.float32))
        hd = TTensor(rows0, self.conv1.cout, dev)
        hd.buf.copy_(h.buf)
        L.psg_tl_mul(hd.ptr, hd.wchunks, mk.ptr, mk.wchunks, rows0, self.conv1.cout, 2.0, st)
        r2 = self._conv_bn_relu(self.conv2, hd, hd.wchunks, None, 0, rows0)
        z = r2["z"]
        logp = torch.empty(B, N, self.ncls, dtype=torch.float32, device=dev)
        L.psg_log_softmax_rows(z.ptr, z.wchunks, rows0, self.ncls, logp.data_ptr(), st)
        l4 = feats[4].to_channels_first(B, xyzs[4].shape[1], widths[4])
        self.ctx = {"B": B, "N": N, "sa": sa_recs, "fp": fp_recs, "r1": r1, "r2": r2, "mask": mk, "feats": feats, "widths": widths}
        return logp, l4

    # ---- backward ---------------------------------------------------------------------------------
    def backward(self, dlogp: torch.Tensor):
        """dlogp [B,N,ncls] -> {parameter: gradient} for every parameter of the model."""
        c = self.ctx
        if c is None:
            raise RuntimeError("backward() needs the activations of a train-mode forward()")
        self.ctx = None
        dev, st = self.dev, _stream()
        B, N = c["B"], c["N"]
        rows0 = B * N
        grads = {}
        dlogp = dlogp.contiguous()
        z = c["r2"]["z"]
        dz = TTensor(rows0, self.ncls, dev, zero=True)
        L.psg_dlogits_from_dlogp(z.ptr, z.wchunks, dlogp.data_ptr(), rows0, self.ncls, dz.ptr, dz.wchunks, st)
        dh = self._chain_backward([c["r2"]], dz, grads)                       # conv2 (no BN): dz -> d(dropped h)
        L.psg_tl_mul(dh.ptr, dh.wchunks, c["mask"].ptr, c["mask"].wchunks, rows0, self.conv1.cout, 2.0, st)
        top = self._chain_backward([c["r1"]], dh, grads)                      # conv1 + bn1 + relu
        # feature propagation, fine to coarse; dcat of level f holds [d skip | d interpolated]
        dlevel = [None] * 5          # (tensor, wchunks view) of the gradient w.r.t. the level features
        for f in (0, 1, 2, 3):
            fr = c["fp"][f]
            dcat = self._chain_backward(fr["recs"], top, grads)
            Nf, Nc, C1, C2 = fr["Nf"], fr["Nc"], fr["C1"], fr["C2"]
            if f > 0:
                dlevel[f] = dcat                                             # columns [0, C1) are d feats[f]; SA adds to them
            offs, perm = self._csr(fr["nn_idx"], B, Nf * 3, Nc)
            dst = TTensor(B * Nc, C2, dev)
            L.psg_segment_sum(dcat.ptr, dcat.wchunks, C1 // 4, Nf, 3, fr["nn_w"].data_ptr(), offs.data_ptr(), perm.data_ptr(),
                              Nf * 3, Nc, B, C2, dst.ptr, dst.wchunks, 0, 0, st)
            if f < 3:
                top = dst
            else:
                dlevel[4] = dst
        # set abstraction, coarse to fine
        for l in (4, 3, 2, 1):
            sr = c["sa"][l - 1]
            S, R, D = sr["S"], sr["R"], sr["D"]
            dsrc = dlevel[l]
            if getattr(self, "debug", None) is not None:          # tools/train_diag.py
                tmp = TTensor(1, 16, dev)
                tmp.buf, tmp.cpad, tmp.rows, tmp.rpad = dsrc.buf, dsrc.cpad, dsrc.rows, dsrc.rpad
                self.debug[l] = tmp.to_channels_first(B, S, c["widths"][l], 0)
            for bi, br in enumerate(sr["branches"]):
                K, cw = br["K"], br["cw"]
                rows = B * S * K
                dy = TTensor(rows, cw, dev)
                L.psg_group_max_backward(dsrc.ptr, dsrc.wchunks, br["col"] // 4, sr["out"].ptr, sr["out"].wchunks, br["col"] // 4,
                                         br["arg"].data_ptr(), B * S, K, cw, dy.ptr, dy.wchunks, st)
                dG = self._chain_backward(br["recs"], dy, grads, need_input_grad=(l > 1))
                if l > 1:
                    # every slot counts here: BatchNorm's backward makes the gradient rows of the padded slots (copies of
                    # the first hit) non-zero, unlike in the eval-mode path where only arg-max rows carry gradient
                    offs, perm = self._csr(br["idx"], B, S * K, R, pad_group=0)
                    tgt = dlevel[l - 1]
                    L.psg_segment_sum(dG.ptr, dG.wchunks, 0, S * K, 1, None, offs.data_ptr(), perm.data_ptr(), S * K, R, B, D,
                                      tgt.ptr, tgt.wchunks, 0, 1, st)
        return grads

    def _csr(self, keys_i32, P, M, R, pad_group=0):
        offs = torch.empty(P * (R + 1), dtype=torch.int32, device=self.dev)
        perm = torch.empty(P * M, dtype=torch.int32, device=self.dev)
        ws = torch.empty(max(L.psg_csr_workspace(P, M, R), 16), dtype=torch.uint8, device=self.dev)
        L.psg_csr_build_by_source(keys_i32.data_ptr(), P, M, R, pad_group, offs.data_ptr(), perm.data_ptr(), ws.data_ptr(), _stream())
        return offs, perm


# ------------------------------------------------------------------------------------------------------
# autograd entry (the reference's own training loop: train_semseg.py:164-179)
# ------------------------------------------------------------------------------------------------------
class _TrainFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, model, *params):
        eng = train_engine(model)
        with torch.cuda.device(x.device):
            logp, l4 = eng.forward(x, getattr(model, "_dropout_mask", None), getattr(model, "_fps_starts", None))
        ctx.eng, ctx.params = eng, params
        ctx.saved_ctx = eng.ctx
        ctx.mark_non_differentiable(l4)
        return logp, l4

    @staticmethod
    def backward(ctx, dlogp, dl4):
        eng = ctx.eng
        eng.ctx = ctx.saved_ctx
        with torch.cuda.device(dlogp.device):
            grads = eng.backward(dlogp)
        return (None, None) + tuple(grads.get(p) for p in ctx.params)


def train_engine(model, mlp_mode=None) -> TrainEngine:
    eng = model.__dict__.get("_psg_train_engine")
    mode = model.__dict__.get("train_mlp_mode", MLP_FP32) if mlp_mode is None else mlp_mode
    if eng is None or eng.mode != mode or eng.dev != next(model.parameters()).device:
        eng = TrainEngine(model, mode)
        model.__dict__["_psg_train_engine"] = eng
    return eng


def train_forward(model, x):
    """``model.train()(x)``: (logp, l4_points) with gradients flowing to the parameters."""
    params = [p for p in model.parameters()]
    out = _TrainFn.apply(x, model, *params)
    invalidate_eval_caches(model)
    return out


def invalidate_eval_caches(model):
    """Parameters / running statistics were (or are about to be) changed through raw pointers: drop the folded eval-mode
    engines built from the old values."""
    if hasattr(model, "_engine"):
        model._engine, model._engine_key = None, None
    for m in model.modules():
        m.__dict__.pop("_psg_chains", None)


# ------------------------------------------------------------------------------------------------------
# weighted NLL as its own differentiable op (get_loss, pointnet2_sem_seg.py:43-49)
# ------------------------------------------------------------------------------------------------------
class _NllFn(torch.autograd.Function):
    @staticmethod
    @L.on_device_of
    def forward(ctx, pred, target, weight):
        pred_c = pred.contiguous()
        rows, ncls = pred_c.shape
        tgt = target.to(device=pred.device, dtype=torch.int64).contiguous()
        w = weight.to(device=pred.device, dtype=torch.float32).contiguous() if weight is not None else None
        out = torch.empty(2, dtype=torch.float32, device=pred.device)
        ws = torch.empty(L.psg_nll_workspace(), dtype=torch.uint8, device=pred.device)
        L.psg_nll_loss(pred_c.data_ptr(), tgt.data_ptr(), w.data_ptr() if w is not None else None, rows, ncls, out.data_ptr(),
                       out[1:].data_ptr(), ws.data_ptr(), ws.numel(), _stream())
        ctx.saved = (tgt, w, out, rows, ncls)
        return out[0]

    @staticmethod
    @L.on_device_of
    def backward(ctx, g):
        tgt, w, out, rows, ncls = ctx.saved
        d = torch.empty(rows, ncls, dtype=torch.float32, device=g.device)
        gc = g.contiguous().float()
        L.psg_nll_loss_backward(tgt.data_ptr(), w.data_ptr() if w is not None else None, rows, ncls, gc.data_ptr(),
                                out[1:].data_ptr(), d.data_ptr(), _stream())
        return d, None, None


def nll_loss(pred, target, weight=None):
    """F.nll_loss(pred, target, weight=weight) for CUDA log-probabilities [rows, ncls]."""
    if not pred.is_cuda:
        raise RuntimeError("pointsecguard_b200.train.nll_loss needs CUDA tensors; there is no CPU fallback")
    return _NllFn.apply(pred, target, weight)


# ------------------------------------------------------------------------------------------------------
# the whole step without autograd in between
# ------------------------------------------------------------------------------------------------------
class Trainer:
    """train_semseg.py:164-179 as one call: forward (train mode), weighted NLL, backward, Adam (:125-132)."""

    def __init__(self, model, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-4, mlp_mode: int = MLP_FP32):
        self.model = model
        self.eng = TrainEngine(model, mlp_mode)
        self.lr, self.betas, self.eps, self.wd = float(lr), (float(betas[0]), float(betas[1])), float(eps), float(weight_decay)
        self.params = [p for p in model.parameters()]
        dev = self.eng.dev
        n = sum(p.numel() for p in self.params)
        # one flat buffer: the parameters become views of it, so Adam is ONE kernel over n elements
        self.flat = torch.empty(n, dtype=torch.float32, device=dev)
        self.flat_grad = torch.zeros(n, dtype=torch.float32, device=dev)
        self.exp_avg = torch.zeros(n, dtype=torch.float32, device=dev)
        self.exp_avg_sq = torch.zeros(n, dtype=torch.float32, device=dev)
        self.offsets = {}
        off = 0
        for p in self.params:
            k = p.numel()
            self.flat[off:off + k].copy_(p.data.reshape(-1))
            p.data = self.flat[off:off + k].view(p.shape)
            self.offsets[p] = (off, k)
            off += k
        self.step_count = 0
        self._out = torch.empty(2, dtype=torch.float32, device=dev)
        self._nll_ws = torch.empty(L.psg_nll_workspace(), dtype=torch.uint8, device=dev)

    def set_lr(self, lr):
        self.lr = float(lr)

    def loss_and_grads(self, x, target, weight=None, dropout_mask=None, starts=None):
        """One train-mode forward + backward.  Returns (loss [device scalar], logp); gradients land in ``flat_grad``
        (``grad_of(p)`` views them per parameter)."""
        dev = self.eng.dev
        with torch.cuda.device(dev):
            st = _stream()
            self.model.train()
            logp, _ = self.eng.forward(x, dropout_mask, starts)
            rows, ncls = logp.shape[0] * logp.shape[1], logp.shape[2]
            tgt = target.to(device=dev, dtype=torch.int64).contiguous().view(-1)
            w = weight.to(device=dev, dtype=torch.float32).contiguous() if weight is not None else None
            L.psg_nll_loss(logp.data_ptr(), tgt.data_ptr(), w.data_ptr() if w is not None else None, rows, ncls,
                           self._out.data_ptr(), self._out[1:].data_ptr(), self._nll_ws.data_ptr(), self._nll_ws.numel(), st)
            dlogp = torch.empty_like(logp)
            L.psg_nll_loss_backward(tgt.data_ptr(), w.data_ptr() if w is not None else None, rows, ncls, None,
                                    self._out[1:].data_ptr(), dlogp.data_ptr(), st)
            grads = self.eng.backward(dlogp)
            for p, (off, k) in self.offsets.items():
                g = grads.get(p)
                if g is None:
                    self.flat_grad[off:off + k].zero_()
                else:
                    self.flat_grad[off:off + k].copy_(g.reshape(-1))
            return self._out[0].clone(), logp

    def grad_of(self, p):
        off, k = self.offsets[p]
        return self.flat_grad[off:off + k].view(p.shape)

    def step(self, x, target, weight=None, dropout_mask=None, starts=None):
        loss, logp = self.loss_and_grads(x, target, weight, dropout_mask, starts)
        self.apply_adam()
        return loss, logp

    def apply_adam(self):
        self.step_count += 1
        with torch.cuda.device(self.eng.dev):
            L.psg_adam_step(self.flat.data_ptr(), self.flat_grad.data_ptr(), self.exp_avg.data_ptr(), self.exp_avg_sq.data_ptr(),
                            self.flat.numel(), self.lr, self.betas[0], self.betas[1], self.eps, self.wd, self.step_count, _stream())
        invalidate_eval_caches(self.model)
