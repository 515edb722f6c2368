"""Host-side owner of one ``psg_net`` (csrc/net.cu): folds eval-mode BatchNorm into the 1x1 convs,
hands the folded weights to the C library, owns the device workspace and draws the FPS start
indices exactly like the reference does.

Reference: PointNet/models/pointnet2_sem_seg.py:6-40, pointnet2_sem_seg_msg.py:6-41 (architecture),
PointNet/models/pointnet_util.py:75 (``torch.randint`` FPS start on the CPU generator, once per SA
level per forward).
"""
from __future__ import annotations

import contextlib
import ctypes as C
import os
from typing import Dict, List, Sequence

import numpy as np
import torch

from . import _lib as L

def _on_engine_device(fn):
    """Engine methods launch on the engine's device whatever device is current in the caller."""
    import functools

    @functools.wraps(fn)
    def wrapped(self, *args, **kwargs):
        if self.device.index == torch.cuda.current_device():
            return fn(self, *args, **kwargs)
        with torch.cuda.device(self.device):
            return fn(self, *args, **kwargs)

    return wrapped


MLP_FP32 = 0     # CUDA-core fp32 GEMMs (parity mode)
MLP_TF32 = 1     # tcgen05 TF32 tensor-core GEMMs (fused kernels)
MLP_TF32X3 = 2   # tcgen05, error-compensated 3xTF32 per-layer GEMMs: fp32-grade results on the tensor cores


def fold_conv_bn(w: torch.Tensor, b: torch.Tensor, bn: Dict[str, torch.Tensor] | None, eps: float = 1e-5):
    """conv(1x1) followed by eval-mode BatchNorm as one affine map, folded in float64."""
    w2 = w.detach().double().cpu().reshape(w.shape[0], w.shape[1])
    b2 = b.detach().double().cpu() if b is not None else torch.zeros(w.shape[0], dtype=torch.float64)
    if bn is not None:
        scale = bn["weight"].detach().double().cpu() / torch.sqrt(bn["running_var"].detach().double().cpu() + eps)
        w2 = w2 * scale[:, None]
        b2 = (b2 - bn["running_mean"].detach().double().cpu()) * scale + bn["bias"].detach().double().cpu()
    return w2.float().contiguous().numpy(), b2.float().contiguous().numpy()


class Engine:
    """One bound network.  ``layers`` is the architecture description produced by the model
    classes (models/pointnet2_sem_seg*.py):

        {"in_channels": 9, "num_classes": 13,
         "sa": [{"npoint", "radius": [..], "nsample": [..], "mlps": [[(w, b), ...], ...]}, ...] x4,
         "fp": [[(w, b), ...] for fp1, fp2, fp3, fp4],      # fine -> coarse
         "conv1": (w, b), "conv2": (w, b)}

    where every (w, b) is already folded and the first SA layer's input columns are ordered
    [features | xyz].
    """

    def __init__(self, layers: dict, device: torch.device, mlp_mode: int = MLP_FP32):
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("pointsecguard_b200 runs on CUDA devices only (no CPU fallback)")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self._keep: List[np.ndarray] = []
        if any(len(sa["mlps"]) > 2 or any(len(m) > 3 for m in sa["mlps"]) for sa in layers["sa"]) or \
                any(len(m) > 3 for m in layers["fp"]):
            raise L.PsgError("psg_net_create takes at most 2 branches per SA level and 3 layers per branch and FP level")
        d = L.NetDesc()
        d.in_channels = layers["in_channels"]
        d.num_classes = layers["num_classes"]
        d.mlp_mode = mlp_mode
        for li, sa in enumerate(layers["sa"]):
            s = d.sa[li]
            s.npoint = sa["npoint"]
            s.nbranch = len(sa["radius"])
            for bi in range(s.nbranch):
                s.radius[bi] = float(sa["radius"][bi])
                s.nsample[bi] = int(sa["nsample"][bi])
                s.nlayers[bi] = len(sa["mlps"][bi])
                for j, (w, b) in enumerate(sa["mlps"][bi]):
                    self._fill(s.mlp[bi][j], w, b)
        for fi, mlps in enumerate(layers["fp"]):
            f = d.fp[fi]
            f.nlayers = len(mlps)
            for j, (w, b) in enumerate(mlps):
                self._fill(f.mlp[j], w, b)
        self._fill(d.conv1, *layers["conv1"])
        self._fill(d.conv2, *layers["conv2"])
        self.npoints = [sa["npoint"] for sa in layers["sa"]]
        self._nsample = [list(sa["nsample"]) for sa in layers["sa"]]
        self.num_classes = layers["num_classes"]
        self.in_channels = layers["in_channels"]
        self.c4 = sum(m[-1][0].shape[0] for m in layers["sa"][3]["mlps"])
        with torch.cuda.device(self.device):
            self._net = L.psg_net_create(C.byref(d))
        self._keep.clear()
        if not self._net:
            raise L.PsgError("psg_net_create failed (unsupported architecture or out of device memory)")
        self.B = self.N = self.T = 0
        self._ws = None
        self.mlp_mode = mlp_mode
        self.shard = None           # distributed.Shard when the bound batch is a slice of a global batch
        self._stream_handle = None
        self._stream_obj = None

    def _fill(self, m: L.MlpDesc, w: np.ndarray, b: np.ndarray):
        w = np.ascontiguousarray(w, dtype=np.float32)
        b = np.ascontiguousarray(b, dtype=np.float32)
        self._keep += [w, b]
        m.cout, m.cin = w.shape
        m.w_host = w.ctypes.data
        m.b_host = b.ctypes.data

    def __del__(self):
        net, self._net = getattr(self, "_net", None), None
        destroy = getattr(L, "psg_net_destroy", None)      # module globals may already be gone at interpreter exit
        if net and destroy is not None:
            destroy(net)

    # ------------------------------------------------------------------------------------------
    def set_mlp_mode(self, mode: int):
        L.psg_net_set_mlp_mode(self._net, mode)
        self.mlp_mode = mode

    @_on_engine_device
    def bind(self, B: int, N: int, T: int):
        """(Re)allocate the workspace for B blocks of N points and T forwards' worth of geometry."""
        if (B, N) == (self.B, self.N) and T <= self.T:
            return
        need = L.psg_net_workspace(self._net, B, N, T)
        if need == 0:
            raise L.PsgError("psg_net_workspace: invalid problem size")
        self._ws = None
        # PSG_GUARD=<MiB>: guard bands of a known byte pattern around the workspace (tests/test_gpu_guard.py checks them
        # after whole attacks -- the pool's compute-sanitizer is closed, so out-of-bounds writes are hunted this way)
        guard = int(os.environ.get("PSG_GUARD", "0")) << 20
        self._guard = guard
        self._ws = torch.empty(need + 1024 + 2 * guard, dtype=torch.uint8, device=self.device)
        if guard:
            self._ws.fill_(0xA5)
        base = (self._ws.data_ptr() + guard + 1023) & ~1023
        self._ws_span = (base - self._ws.data_ptr(), need)
        L.psg_net_bind(self._net, B, N, T, base, need)
        self.B, self.N, self.T = B, N, T

    def guard_intact(self) -> bool:
        """True when the guard bands around the workspace (PSG_GUARD) still hold their pattern."""
        if not getattr(self, "_guard", 0) or self._ws is None:
            return True
        off, need = self._ws_span
        head = self._ws[:off]
        tail = self._ws[off + need:]
        return bool((head == 0xA5).all().item()) and bool((tail == 0xA5).all().item())

    def _stream(self):
        """Stream the C library enqueues on: the one set with ``use_stream`` (the geometry head start's tail engine,
        torchattacks/attacks/nontarget.py) or torch's current stream."""
        return self._stream_handle if self._stream_handle is not None else torch.cuda.current_stream(self.device).cuda_stream

    def set_xyz_grad(self, on: bool):
        """Also produce the geometric gradient w.r.t. coordinates (csrc/geomgrad.cu) in backward()."""
        L.psg_net_set_xyz_grad(self._net, 1 if on else 0)

    def use_stream(self, stream):
        """Pin this engine to a torch.cuda.Stream (None = follow torch's current stream)."""
        self._stream_handle = stream.cuda_stream if stream is not None else None
        self._stream_obj = stream

    def draw_starts(self, T: int) -> torch.Tensor:
        """FPS start indices for T forwards, drawn on the global CPU generator in the reference's
        call order (per forward: level 1..4, each ``torch.randint(0, N_level, (B,))``,
        pointnet_util.py:75).  Returns int32 [4, T, B] (CPU)."""
        from .distributed import Shard, draw_starts
        sizes = [self.N] + self.npoints[:3]
        shard = self.shard if self.shard is not None else Shard(self.B, 0, self.B)
        if shard.size != self.B:
            raise ValueError(f"shard of {shard.size} blocks does not match the bound batch of {self.B}")
        return draw_starts(sizes, T, shard)

    def set_shard(self, shard):
        """Declare the bound batch to be ``shard`` of a global batch (multi-GPU runs): the FPS start
        draws are then made for the whole global batch and sliced, so every rank consumes the CPU
        generator like the single-GPU run does."""
        self.shard = shard

    @_on_engine_device
    def set_input(self, x: torch.Tensor):
        if x.dim() != 3 or x.shape[0] != self.B or x.shape[1] != self.in_channels or x.shape[2] != self.N:
            raise ValueError(f"expected [{self.B},{self.in_channels},{self.N}], got {tuple(x.shape)}")
        if x.dtype != torch.float32 or x.device != self.device:
            raise TypeError("input must be a float32 tensor on the engine's CUDA device")
        sb, sc, sn = x.stride()
        L.psg_net_set_input(self._net, x.data_ptr(), sb, sc, sn, self._stream())

    @_on_engine_device
    def copy_input_from(self, other: "Engine"):
        """Take over the packed model input of ``other`` (same B, N): the colours as its last update projected them."""
        rc = L.psg_net_copy_input(self._net, other._net, self._stream())
        if rc != 0:
            raise L.PsgError(f"psg_net_copy_input failed ({rc})")

    @_on_engine_device
    def geometry(self, starts: torch.Tensor):
        """starts: int32 [4, T, B] (CPU or device)."""
        T = starts.shape[1]
        if T > self.T or starts.shape[2] != self.B:
            raise ValueError("geometry: starts do not match the bound problem")
        # the upload is enqueued on the stream the FPS kernels read it on (a pinned engine's side stream: the block then
        # belongs to that stream in the caching allocator, so replacing the previous chunk's starts is stream-ordered too)
        with torch.cuda.stream(self._stream_obj) if self._stream_obj is not None else contextlib.nullcontext():
            self._starts_dev = starts.to(device=self.device, dtype=torch.int32, non_blocking=True).contiguous()
        L.psg_net_geometry(self._net, self._starts_dev.data_ptr(), T, self._stream())

    @_on_engine_device
    def read_geometry(self, what: str, level: int, branch: int = 0, t: int = 0) -> torch.Tensor:
        """The resident index buffers the network forward consumes (slot t): ``what`` in fps | ball | nn_idx | nn_w |
        xyz; SA levels 1..4, FP levels 0 (fp1) .. 3 (fp4).  Parity tests compare them with the oracle."""
        code = {"fps": 0, "ball": 1, "nn_idx": 2, "nn_w": 3, "xyz": 4}[what]
        np_ = [self.N] + self.npoints
        if code == 0:
            out = torch.empty(self.B, np_[level], dtype=torch.int32, device=self.device)
        elif code == 4:
            out = torch.empty(self.B, np_[level], 3, dtype=torch.float32, device=self.device)
        elif code == 1:
            out = torch.empty(self.B, np_[level], self._nsample[level - 1][branch], dtype=torch.int32, device=self.device)
        else:
            out = torch.empty(self.B, np_[level], 3, dtype=torch.int32 if code == 2 else torch.float32, device=self.device)
        L.psg_net_read_geometry(self._net, code, level, branch, t, out.data_ptr(), out.numel() * 4, self._stream())
        return out

    @_on_engine_device
    def forward(self, t: int = 0, want_logp: bool = True, want_l4: bool = False):
        logp = torch.empty(self.B, self.N, self.num_classes, dtype=torch.float32, device=self.device) if want_logp else None
        l4 = torch.empty(self.B, self.c4, self.npoints[3], dtype=torch.float32, device=self.device) if want_l4 else None
        L.psg_net_forward(self._net, t, logp.data_ptr() if want_logp else None, l4.data_ptr() if want_l4 else None,
                          self._stream())
        return logp, l4

    @_on_engine_device
    def loss_grad_generic(self, dlogp: torch.Tensor):
        dlogp = dlogp.contiguous()
        self._dlogp_keep = dlogp      # read by the kernels psg_net_backward launches (deferred loss, tcgen05 mode)
        L.psg_net_loss_grad(self._net, 0, dlogp.data_ptr(), None, -1, 1.0, 0.0, None, self._stream())

    @_on_engine_device
    def loss_grad_ce(self, labels: torch.Tensor | None, target: int, scale: float):
        L.psg_net_loss_grad(self._net, 1, None, labels.data_ptr() if labels is not None else None, target, scale, 0.0,
                            None, self._stream())

    @_on_engine_device
    def loss_grad_cw(self, labels: torch.Tensor | None, target: int, sign: float, kappa: float, loss_rows=None):
        L.psg_net_loss_grad(self._net, 2, None, labels.data_ptr() if labels is not None else None, target, sign, kappa,
                            loss_rows.data_ptr() if loss_rows is not None else None, self._stream())

    @_on_engine_device
    def backward(self, t: int = 0, want_grad: bool = True):
        g = torch.empty(self.B, self.in_channels, self.N, dtype=torch.float32, device=self.device) if want_grad else None
        L.psg_net_backward(self._net, t, g.data_ptr() if want_grad else None, self._stream())
        return g

    @_on_engine_device
    def pgd_update(self, adv, ori, mask, c0, nc, alpha_signed, eps, lo=0.0, hi=1.0):
        L.psg_net_pgd_update(self._net, adv.data_ptr(), ori.data_ptr(), mask.data_ptr() if mask is not None else None,
                             c0, nc, alpha_signed, eps, lo, hi, self._stream())

    @_on_engine_device
    def pgd_update_l2(self, adv, ori, mask, c0, nc, alpha_signed, eps, lo=0.0, hi=1.0):
        """``pgd_update`` with torchattacks PGDL2's step and L2-ball projection, per block over its moving points."""
        L.psg_net_pgd_update_l2(self._net, adv.data_ptr(), ori.data_ptr(), mask.data_ptr() if mask is not None else None,
                                c0, nc, alpha_signed, eps, lo, hi, self._stream())

    @_on_engine_device
    def nb_attack(self, adv, ori, mask, labels, target, iters, t0, alpha, eps, scale, norm="Linf"):
        """``iters`` NB / tar-NB iterations from forward slot t0; ``norm`` "Linf" (sign step) or "L2" (PGDL2 step)."""
        if norm not in ("Linf", "L2"):
            raise ValueError(f"norm must be 'Linf' or 'L2', got {norm!r}")
        fn = L.psg_nb_attack if norm == "Linf" else L.psg_nb_attack_l2
        fn(self._net, adv.data_ptr(), ori.data_ptr(), mask.data_ptr() if mask is not None else None,
           labels.data_ptr() if labels is not None else None, target, iters, t0, alpha, eps, scale, self._stream())
