"""Dense dilated kNN graph -- drop-in for ResGCN/gcn_lib/dense/torch_edge.py:6-81 (SURVEY.md section 8f rank 4).

``dense_knn_matrix`` is the hot op of ResGCN's dynamic graph (one call per block of the network): the reference builds the
full [B, N, N] distance matrix and runs ``torch.topk`` over it; here ``psg_dense_knn`` (csrc/knn.cu) streams the cloud
through shared memory and keeps each query's best k on chip, so no distance reaches HBM.  Any feature width C and any
k * dilation up to min(N, 1024) neighbours: every dilated graph of ResGCN-28 (k * dilation = 16 ... 432).
Same names, signatures and tensor conventions (x [B, C, N, 1] -> edge_index [2, B, N, k]); CUDA tensors only, no CPU
fallback.  Order: nearest first, exact ties by ascending index; NaN distances (NaN or infinite features) come after +inf,
whereas ``torch.topk`` ranks NaN first -- so every index is in [0, N) and appears once per row.  The sparse
``DilatedKnnGraph`` (torch_cluster) and the ResGCN model / its colour attacks are outside this repository's scope.
"""
from __future__ import annotations

import torch
from torch import nn

from ... import _lib as L

MAX_K = 1024          # the most neighbours psg_dense_knn returns per point

def _stream():
    return torch.cuda.current_stream().cuda_stream


class DenseDilated(nn.Module):
    """torch_edge.py:6-29: every ``dilation``-th neighbour of the list (or a random subset when stochastic)."""

    def __init__(self, k=9, dilation=1, stochastic=False, epsilon=0.0):
        super().__init__()
        self.dilation = dilation
        self.stochastic = stochastic
        self.epsilon = epsilon
        self.k = k

    def forward(self, edge_index):
        if self.stochastic:
            if torch.rand(1) < self.epsilon and self.training:
                num = self.k * self.dilation
                randnum = torch.randperm(num)[:self.k]
                edge_index = edge_index[:, :, :, randnum]
            else:
                edge_index = edge_index[:, :, :, ::self.dilation]
        else:
            edge_index = edge_index[:, :, :, ::self.dilation]
        return edge_index


@L.on_device_of
def pairwise_distance(x):
    """torch_edge.py:32-43: x [B, N, C] -> squared distances [B, N, N] (x_square + (-2 x x^T) + x_square^T)."""
    if not x.is_cuda:
        raise RuntimeError("pointsecguard_b200.gcn_lib runs on CUDA tensors only; there is no CPU fallback")
    xc = x.detach().float().contiguous()
    B, N, C = xc.shape
    out = torch.empty(B, N, N, dtype=torch.float32, device=x.device)
    L.psg_pairwise_distance(xc.data_ptr(), B, N, C, out.data_ptr(), _stream())
    return out


@L.on_device_of
def dense_knn_matrix(x, k=16):
    """torch_edge.py:45-59: x [B, C, N, 1] -> stack((nn_idx, center_idx)) [2, B, N, k] (long); 1 <= k <= min(N, 1024)."""
    if not x.is_cuda:
        raise RuntimeError("pointsecguard_b200.gcn_lib runs on CUDA tensors only; there is no CPU fallback")
    with torch.no_grad():
        xc = x.detach().transpose(2, 1).squeeze(-1).float().contiguous()          # [B, N, C]
        B, N, C = xc.shape
        if not 1 <= k <= min(N, MAX_K):
            raise ValueError(f"dense_knn_matrix: k = {k} neighbours requested, but k must lie in [1, min(N, {MAX_K})] "
                             f"with N = {N} points")
        nn_idx = torch.empty(B, N, k, dtype=torch.int64, device=x.device)
        L.psg_dense_knn(xc.data_ptr(), B, N, C, int(k), nn_idx.data_ptr(), None, _stream())
        center_idx = torch.arange(0, N, device=x.device).repeat(B, k, 1).transpose(2, 1)
    return torch.stack((nn_idx, center_idx), dim=0)


class DenseDilatedKnnGraph(nn.Module):
    """torch_edge.py:62-81: k * dilation nearest neighbours, then the dilated selection."""

    def __init__(self, k=9, dilation=1, stochastic=False, epsilon=0.0):
        super().__init__()
        self.dilation = dilation
        self.stochastic = stochastic
        self.epsilon = epsilon
        self.k = k
        self._dilated = DenseDilated(k, dilation, stochastic, epsilon)
        self.knn = dense_knn_matrix

    def forward(self, x):
        edge_index = self.knn(x, self.k * self.dilation)
        return self._dilated(edge_index)
