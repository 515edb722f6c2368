"""Dense kNN graph at any feature width and up to 1024 neighbours (csrc/knn.cu, DESIGN.md section 12).

Exact selection: ``psg_dense_knn`` computes every distance with the recipe of ``psg_pairwise_distance``, so its output must
equal, index for index and bit for bit, the first k columns of a stable (distance, index) sort of the pairwise-distance rows
with NaN after +inf.  Reference parity at ResGCN-28's shapes uses the rule of tests/test_knn.py: a differing neighbour slot is
accepted only where the two candidates' distances agree to rounding."""
import numpy as np
import pytest
import torch

from oracle import knn_oracle as KO
from pointsecguard_b200 import synthetic as syn

RESGCN_K, RESGCN_BLOCKS = 16, 27           # ResGCN-28: k = 16, backbone block i dilated by 1 + i


def _features(B, N, C, kind, seed):
    """[B, N, C] features from synthetic blocks: the 9 block channels (grid: the 3 grid coordinates) repeated to C, so that
    exact ties and duplicate points survive at every width."""
    kind = kind if N > 1 else "uniform"                                             # one point has no duplicate
    blk = syn.make_blocks(B, N, seed, kind).transpose(2, 1).contiguous()           # [B, N, 9]
    src = blk[..., :3] if kind == "grid" else blk
    reps = (C + src.shape[-1] - 1) // src.shape[-1]
    return src.repeat(1, 1, reps)[..., :C].contiguous()


def _knn(x, k):
    """psg_dense_knn on x [B, N, C] (CUDA): (idx [B,N,k] int64, d2 [B,N,k])."""
    from pointsecguard_b200 import _lib as L
    B, N, C = x.shape
    idx = torch.empty(B, N, k, dtype=torch.int64, device=x.device)
    d2 = torch.empty(B, N, k, dtype=torch.float32, device=x.device)
    L.psg_dense_knn(x.data_ptr(), B, N, C, k, idx.data_ptr(), d2.data_ptr(), torch.cuda.current_stream().cuda_stream)
    return idx, d2


def _stable_order(d):
    """Indices sorting each row of d by (distance, index), NaN after +inf."""
    nan = torch.isnan(d)
    o1 = torch.sort(torch.where(nan, torch.full_like(d, float("inf")), d), dim=-1, stable=True)[1]
    o2 = torch.sort(nan.gather(-1, o1).to(torch.int8), dim=-1, stable=True)[1]
    return o1.gather(-1, o2)


def _assert_exact(x, idx, d2, rows=None):
    """idx / d2 [B, N, k] (or [B, len(rows), k] for the query rows ``rows``) against the stable sort of pairwise_distance."""
    from pointsecguard_b200.gcn_lib.dense import pairwise_distance
    k = idx.shape[-1]
    d = pairwise_distance(x)
    if rows is not None:
        d = d[:, rows]
    want = _stable_order(d)[..., :k]
    assert torch.equal(idx, want), f"first mismatch at {torch.nonzero(idx != want)[0].tolist()}"
    if d2 is not None:
        g = d.gather(-1, want)
        assert torch.equal(torch.isnan(d2), torch.isnan(g))
        assert torch.equal(torch.nan_to_num(d2), torch.nan_to_num(g))


EXACT_C = [1, 3, 9, 64, 65, 128, 200, 1024]
KINDS = ["uniform", "grid", "duplicates", "clustered"]


@pytest.mark.gpu
@pytest.mark.parametrize("C", EXACT_C)
def test_exact_selection(C):
    n_calls = 0
    for ni, N in enumerate([1, 33, 1000, 4096]):
        for ki, k in enumerate([1, 33, 100, 432, 1024]):
            if k > N:
                continue
            B = 3 if (ni + ki) % 2 else 1
            kind = KINDS[(ni + ki + EXACT_C.index(C)) % 4]
            x = _features(B, N, C, kind, seed=100 * ni + ki).cuda()
            idx, d2 = _knn(x, k)
            assert idx.shape == (B, N, k)
            _assert_exact(x, idx, d2)
            n_calls += 1
    assert n_calls == 12


@pytest.mark.gpu
@pytest.mark.parametrize("C", [3, 64])
@pytest.mark.parametrize("kind", ["uniform", "grid"])
def test_prefix_seam(C, kind):
    """k <= 16 (register kernel at C <= 64) and k = 17 ... 33 (shared-memory list kernel) against the first columns of k = 432."""
    x = _features(2, 1000, C, kind, seed=7).cuda()
    big_i, big_d = _knn(x, 432)
    for k in [1, 2, 15, 16, 17, 31, 32, 33]:
        i, d = _knn(x, k)
        assert torch.equal(i, big_i[..., :k]), k
        assert torch.equal(d, big_d[..., :k]), k
    _assert_exact(x, big_i, big_d)


def _resgcn_inputs():
    g = torch.Generator().manual_seed(28)
    blk = syn.make_blocks(2, 4096, 28, "uniform").transpose(2, 1).contiguous()     # [2, 4096, 9]
    w = torch.randn(9, 64, generator=g) / 3.0
    bias = torch.randn(64, generator=g) * 0.1
    return [("randn64", torch.randn(2, 4096, 64, generator=g)),
            ("relu64", torch.relu(blk @ w + bias))]                                # many exact zeros


def _check_against(mine, ref, dref, sq, what):
    """Neighbour slots equal, except where the two candidates' distances agree to 1e-5 relative (plus the rounding of
    |x|^2 that the reference's sgemm and the kernel's fma chain leave at different places)."""
    bad = mine != ref
    if not bad.any():
        return 0
    da, db = dref.gather(-1, mine), dref.gather(-1, ref)
    scale = sq.unsqueeze(-1) + torch.maximum(sq.gather(-1, mine.flatten(1)).view_as(mine),
                                             sq.gather(-1, ref.flatten(1)).view_as(ref))
    tol = 1e-5 * torch.maximum(torch.maximum(da.abs(), db.abs()), torch.full_like(da, 1e-12)) + 4e-7 * scale
    ok = (da - db).abs() <= tol
    assert bool(ok[bad].all()), f"{what}: {int((~ok & bad).sum())} slots differ beyond near-ties"
    return int(bad.sum())


@pytest.mark.gpu
def test_reference_parity_resgcn28():
    from pointsecguard_b200.gcn_lib.dense import DenseDilatedKnnGraph, dense_knn_matrix
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        head = syn.make_blocks(2, 4096, 3, "uniform")[:, :3].transpose(2, 1).contiguous()
        cases = [("xyz", head, [RESGCN_K])] + [(n, f, [RESGCN_K * (1 + i) for i in range(RESGCN_BLOCKS)])
                                               for n, f in _resgcn_inputs()]
        for name, xt, ks in cases:
            xt = xt.cuda()
            x = xt.transpose(2, 1).unsqueeze(-1)                                     # [B, C, N, 1]
            dref = KO.pairwise_distance(xt)
            sq = (xt * xt).sum(-1)
            for kd in ks:
                ref = torch.topk(-dref, k=kd)[1]
                e = dense_knn_matrix(x, kd)
                nbad = _check_against(e[0], ref, dref, sq, f"{name} k={kd}")
                if name == "xyz":
                    assert nbad <= 1e-3 * ref.numel(), nbad
                dil = kd // RESGCN_K
                ed = DenseDilatedKnnGraph(RESGCN_K, dil)(x)
                _check_against(ed[0], ref[..., ::dil], dref, sq, f"{name} dilated {dil}")
                assert torch.equal(ed[1], torch.arange(4096, device="cuda").view(1, -1, 1).expand(2, -1, RESGCN_K))
        # the golden-pinned oracle itself (CPU, reference ops) at the head's k, against the kernel
        xt = head
        e_cpu = KO.dense_knn_matrix(xt.transpose(2, 1).unsqueeze(-1), RESGCN_K)
        e = dense_knn_matrix(xt.cuda().transpose(2, 1).unsqueeze(-1), RESGCN_K).cpu()
        _check_against(e[0], e_cpu[0], KO.pairwise_distance(xt), (xt * xt).sum(-1), "xyz vs CPU oracle")
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev


@pytest.mark.gpu
@pytest.mark.parametrize("C", [64, 1024])
def test_at_size(C):
    """B = 16 clouds of 4096 points: every dilated graph of ResGCN-28 (C = 64), the deepest one at C = 1024; exact selection on
    a seeded subset of query rows of every cloud, and two runs bit-identical."""
    from pointsecguard_b200.gcn_lib.dense import DenseDilatedKnnGraph, pairwise_distance
    g = torch.Generator().manual_seed(16 + C)
    x = torch.randn(16, 4096, C, generator=g).cuda()
    rows = torch.randperm(4096, generator=g)[:48].cuda()
    want_all = _stable_order(pairwise_distance(x)[:, rows])
    dils = range(1, RESGCN_BLOCKS + 1) if C == 64 else [RESGCN_BLOCKS]
    for dil in dils:
        kd = RESGCN_K * dil
        idx, d2 = _knn(x, kd)
        assert torch.equal(idx[:, rows], want_all[..., :kd]), kd
        idx2, d22 = _knn(x, kd)
        assert torch.equal(idx, idx2) and torch.equal(d2, d22), kd
        ed = DenseDilatedKnnGraph(RESGCN_K, dil)(x.transpose(2, 1).unsqueeze(-1))
        assert torch.equal(ed[0], idx[..., ::dil]), kd


@pytest.mark.gpu
@pytest.mark.parametrize("k", [16, 32, 100, 1000])
def test_non_finite(k):
    """NaN / +inf / -inf features: indices in [0, N), unique per row, and the (distance, index) order with NaN last --
    so the finite neighbours come first, in exact order."""
    N = 1000
    x = _features(2, N, 9, "uniform", seed=5)
    x[0, 3, 1] = float("nan")
    x[0, 10, :] = float("inf")
    x[1, 20, 4] = float("-inf")
    x[1, 21, 0] = float("inf")
    x[1, 999, 8] = float("nan")
    x = x.cuda()
    idx, d2 = _knn(x, k)
    assert int(idx.min()) >= 0 and int(idx.max()) < N
    s = idx.sort(-1)[0]
    assert bool((s[..., 1:] != s[..., :-1]).all())
    _assert_exact(x, idx, d2)
    # a finite query sees the non-finite points last
    for b, bad in [(0, {3, 10}), (1, {20, 21, 999})]:
        row = idx[b, 500].tolist()
        n_finite = min(k, N - len(bad))
        assert not set(row[:n_finite]) & bad


@pytest.mark.gpu
def test_error_contract():
    from pointsecguard_b200 import _lib as L
    from pointsecguard_b200.gcn_lib.dense import dense_knn_matrix
    x = torch.rand(1, 8, 2000, 1, device="cuda")
    with pytest.raises(ValueError, match=r"k = 1025.*1024.*N = 2000"):
        dense_knn_matrix(x, 1025)
    with pytest.raises(ValueError, match=r"k = 41.*N = 40"):
        dense_knn_matrix(x[:, :, :40], 41)
    xt = x.squeeze(-1).transpose(2, 1).contiguous()
    out = torch.empty(1, 2000, 1025, dtype=torch.int64, device="cuda")
    with pytest.raises(L.PsgError, match="invalid argument"):
        L.psg_dense_knn(xt.data_ptr(), 1, 2000, 8, 1025, out.data_ptr(), None, torch.cuda.current_stream().cuda_stream)
    with pytest.raises(RuntimeError, match="CUDA tensors only"):
        dense_knn_matrix(x.cpu(), 16)


def test_cpu_tensors_refused_before_k_check():
    """No device needed: CPU tensors are refused by name, whatever k."""
    from pointsecguard_b200.gcn_lib.dense import dense_knn_matrix
    with pytest.raises(RuntimeError, match="CUDA tensors only"):
        dense_knn_matrix(torch.rand(1, 3, 10, 1), 2000)


def test_stable_order_helper():
    """The test's own reference order: (distance, index), NaN after +inf (CPU)."""
    d = torch.tensor([[3.0, float("nan"), 1.0, float("inf"), 1.0, float("nan"), -0.5]])
    assert _stable_order(d).tolist() == [[6, 2, 4, 0, 3, 1, 5]]
    assert np.array_equal(_stable_order(torch.zeros(1, 5)).numpy(), [[0, 1, 2, 3, 4]])
