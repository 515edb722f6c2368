"""Shared forward of the two sem-seg networks: the whole network runs inside one ``psg_net``
(csrc/net.cu) -- geometry, grouped MLPs, feature propagation, head -- and autograd sees it as a
single differentiable op whose backward is the engine's input-gradient pass.
"""
from __future__ import annotations

import torch
import torch.nn as nn

from pointsecguard_b200._lib import on_device_of
from pointsecguard_b200.engine import Engine, MLP_FP32, fold_conv_bn


def _bn_dict(bn):
    return {"weight": bn.weight, "bias": bn.bias, "running_mean": bn.running_mean, "running_var": bn.running_var}


class _NetFn(torch.autograd.Function):
    """(logp, l4_points) = net(x); d x = engine.backward(d logp).  Only the most recent forward
    of an engine can be back-propagated (its activations live in the engine workspace)."""

    @staticmethod
    @on_device_of
    def forward(ctx, x, model, starts):
        eng = model.engine(x.device)
        eng.bind(x.shape[0], x.shape[2], 1)
        eng.set_input(x)
        # decided before the geometry pass: with the coordinate gradient wanted, the set-abstraction rows stay in the padded
        # layout its kernels read (csrc/compact.cu)
        eng.set_xyz_grad(bool(getattr(model, "xyz_grad", False)))
        eng.geometry(starts)
        logp, l4 = eng.forward(0, True, True)
        model._generation += 1
        ctx.model, ctx.gen, ctx.eng = model, model._generation, eng
        ctx.mark_non_differentiable(l4)
        return logp, l4

    @staticmethod
    @on_device_of
    def backward(ctx, dlogp, dl4):
        if ctx.model._generation != ctx.gen:
            raise RuntimeError("pointsecguard_b200: the activations of this forward were overwritten by a later "
                               "forward of the same model; back-propagate before running the model again")
        ctx.eng.loss_grad_generic(dlogp)
        g = ctx.eng.backward(0, True)
        ctx.eng.set_xyz_grad(False)
        return g, None, None


class SemSegBase(nn.Module):
    """get_model.forward of pointnet2_sem_seg.py:22-40 / pointnet2_sem_seg_msg.py:23-41."""

    arch = "ssg"
    # default MLP mode of the eval-mode (attack) engine (set_mlp_mode changes it per model)
    mlp_mode = MLP_FP32
    # autograd of forward(): False = gradient through the features only (all the colour attacks need);
    # True = also through the geometry (centred neighbour coordinates, interpolation weights), which
    # is what the reference's autograd produces on input channels 0:3
    xyz_grad = False

    def _init_runtime(self):
        self._engine = None
        self._engine_key = None
        self._generation = 0
        self._shard = None

    def set_shard(self, shard):
        """Multi-GPU runs: declare that the batches this replica sees are ``shard``
        (pointsecguard_b200.distributed.Shard) of a global batch; FPS start draws are then made for
        the global batch and sliced.  ``None`` restores single-process behaviour."""
        self._shard = shard
        if self._engine is not None:
            self._engine.set_shard(shard)

    # ---- engine management ----------------------------------------------------------------
    def _param_key(self, device):
        items = [(t.data_ptr(), t._version) for t in list(self.parameters()) + list(self.buffers())]
        return (str(device), self.mlp_mode, tuple(items))

    def engine(self, device=None) -> Engine:
        device = torch.device(device) if device is not None else next(self.parameters()).device
        if device.type != "cuda":
            raise RuntimeError("pointsecguard_b200 models run on CUDA devices only; there is no CPU fallback")
        if self.training:
            raise RuntimeError("the folded-BatchNorm engine is the eval-mode (attack) path; train mode runs through "
                               "pointsecguard_b200.train (model.train()(x) or train.Trainer)")
        key = self._param_key(device)
        if self._engine is None or key != self._engine_key:
            self._engine = Engine(self.describe(), device, self.mlp_mode)
            self._engine_key = key
            self._engine.set_shard(self._shard)
        return self._engine

    def tail_engine(self, device, primary=None):
        """A second engine (same folded weights, own workspace) and a side stream: the norm-bounded attacks compute the
        geometry of all but the first forwards on it while the loop already runs (torchattacks/attacks/nontarget.py)."""
        if primary is None:
            primary = self.engine(device)
        if getattr(self, "_tail", None) is None or self._tail_of is not primary:
            self._tail = Engine(self.describe(), primary.device, self.mlp_mode)
            self._tail_of = primary
            self._tail_stream = torch.cuda.Stream(primary.device)
        self._tail.set_mlp_mode(self.mlp_mode)
        return self._tail, self._tail_stream

    def set_mlp_mode(self, mode: int):
        self.mlp_mode = mode
        if self._engine is not None:
            self._engine.set_mlp_mode(mode)
            if getattr(self, "_tail", None) is not None:
                self._tail.set_mlp_mode(mode)
            self._engine_key = self._param_key(self._engine.device)

    def _sa_desc(self, sa):
        """One SA level -> engine description with folded weights, first-layer input columns
        reordered to [features | xyz] (SSG concatenates xyz first, pointnet_util.py:137; MSG
        features first, :253)."""
        if hasattr(sa, "conv_blocks"):
            radii, ks = list(sa.radius_list), list(sa.nsample_list)
            blocks = [(sa.conv_blocks[i], sa.bn_blocks[i]) for i in range(len(radii))]
            xyz_first = False
        else:
            radii, ks = [sa.radius], [sa.nsample]
            blocks = [(sa.mlp_convs, sa.mlp_bns)]
            xyz_first = True
        mlps = []
        for convs, bns in blocks:
            layers = []
            for j, (conv, bn) in enumerate(zip(convs, bns)):
                w, b = fold_conv_bn(conv.weight, conv.bias, _bn_dict(bn), bn.eps)
                if j == 0 and xyz_first:
                    w = w[:, list(range(3, w.shape[1])) + [0, 1, 2]].copy()
                layers.append((w, b))
            mlps.append(layers)
        return {"npoint": sa.npoint, "radius": radii, "nsample": ks, "mlps": mlps}

    def describe(self):
        fps = []
        for fp in (self.fp1, self.fp2, self.fp3, self.fp4):
            fps.append([fold_conv_bn(c.weight, c.bias, _bn_dict(b), b.eps) for c, b in zip(fp.mlp_convs, fp.mlp_bns)])
        return {
            "in_channels": 9,
            "num_classes": self.conv2.out_channels,
            "sa": [self._sa_desc(s) for s in (self.sa1, self.sa2, self.sa3, self.sa4)],
            "fp": fps,
            "conv1": fold_conv_bn(self.conv1.weight, self.conv1.bias, _bn_dict(self.bn1), self.bn1.eps),
            "conv2": fold_conv_bn(self.conv2.weight, self.conv2.bias, None),
        }

    # ---- forward ------------------------------------------------------------------------------
    @on_device_of
    def forward(self, xyz):
        if xyz.dim() != 3 or xyz.shape[1] != 9:
            raise ValueError(f"expected [B, 9, N] input, got {tuple(xyz.shape)}")
        if self.training:
            # train mode (train_semseg.py:168-169): batch-statistics BatchNorm, dropout, gradients to the parameters
            if not xyz.is_cuda:
                raise RuntimeError("pointsecguard_b200 models run on CUDA devices only; there is no CPU fallback")
            from pointsecguard_b200 import train as _train
            return _train.train_forward(self, xyz)
        eng = self.engine(xyz.device)
        eng.bind(xyz.shape[0], xyz.shape[2], 1)
        starts = eng.draw_starts(1)
        return _NetFn.apply(xyz, self, starts)
