"""Sampling and grouping indices on clouds away from the unit box, bit for bit against the C oracle (oracle/geom.py).

Every other geometry test draws its clouds inside about [-0.5, 0.5]^2 x [0, 3] m.  The expansion-form distance
((-2 q.p) + |q|^2) + |p|^2 loses about 2^-24 |p|^2 in absolute terms, so the places where a kernel that only visits
candidates near a query (ball_grid_kernel, three_nn_grid_kernel) can miss a neighbour are clouds far from the origin,
scaled clouds, scene-sized slabs, points exactly on cell boundaries, the grid's fallback seam (96 hits) and non-finite
coordinates.  Ball query is checked through both C entry points -- psg_ball_query_grid (called directly) and
psg_ball_query (the exhaustive scan) -- and through the public op; 3-NN with the grid forced on and off.

The test without a GPU mark restates the grid's candidate set and its margin rule in numpy, so that the reason for the
rule (ballgrid.cu, file comment) can be checked on any machine.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import geom as G
from pointsecguard_b200 import synthetic as syn

gpu = pytest.mark.gpu

RADII = [0.05, 0.1, 0.2, 0.4, 0.8]
OFFSETS = [0.0, 10.0, 50.0, 100.0, 300.0, 1000.0]
# single radius, and MSG pairs in both orders (the grid is binned for the larger one)
RADIUS_SETS = [(r,) for r in RADII] + [(0.1, 0.05), (0.05, 0.1), (0.4, 0.2), (0.2, 0.8)]
# (offset vector, scale): translations on x/y and on z, millimetre and kilometre clouds
TRANSFORMS = [((o, o, 0.0), 1.0) for o in OFFSETS] + [((0.0, 0.0, o), 1.0) for o in OFFSETS[1:]] + \
             [((0.0, 0.0, 0.0), 1e-3), ((0.0, 0.0, 0.0), 1e3)]
TF_IDS = [f"xy{o:g}" for o in OFFSETS] + [f"z{o:g}" for o in OFFSETS[1:]] + ["mm", "km"]


# ---- clouds ---------------------------------------------------------------------------------------------------------
def _block(B, N, seed, offset=(0.0, 0.0, 0.0), scale=1.0):
    """B uniform 1 x 1 x 3 m blocks (the layout of synthetic.make_blocks), scaled, then translated; [B, N, 3] float32."""
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(B, N, 3, generator=g)
    x[..., :2] -= 0.5
    x[..., 2] *= 3.0
    return x * scale + torch.tensor(offset, dtype=torch.float32)


def _pick(xyz, S, seed):
    g = torch.Generator().manual_seed(seed + 1)
    B, N, _ = xyz.shape
    sel = torch.stack([torch.randperm(N, generator=g)[:S] for _ in range(B)])
    return xyz[torch.arange(B)[:, None], sel].contiguous()


def _psg():
    from pointsecguard_b200 import ops  # noqa: F401  (registers torch.ops.psg)
    return torch.ops.psg


# ---- the three ball queries -----------------------------------------------------------------------------------------
def _c_args(radii, ks):
    nr = len(radii)
    return nr, (C.c_double * 2)(*radii, *([0.0] * (2 - nr))), (C.c_int * 2)(*ks, *([0] * (2 - nr)))


def _grid(xyz, new_xyz, radii, ks):
    """psg_ball_query_grid; xyz [nclouds, N, 3], new_xyz [P, S, 3] (problem p reads cloud p % nclouds)."""
    from pointsecguard_b200 import _lib as L
    xyz, new_xyz = xyz.cuda().contiguous(), new_xyz.cuda().contiguous()
    nc, N, _ = xyz.shape
    P, S, _ = new_xyz.shape
    nr, r, k = _c_args(radii, ks)
    outs = [torch.full((P, S, kk), -7, dtype=torch.int32, device="cuda") for kk in ks]
    wsb = L.psg_ball_grid_workspace(nc, N)
    ws = torch.empty(wsb, dtype=torch.uint8, device="cuda")
    L.psg_ball_query_grid(xyz.data_ptr(), nc, P, N, new_xyz.data_ptr(), S, nr, r, k, outs[0].data_ptr(),
                          outs[1].data_ptr() if nr == 2 else None, ws.data_ptr(), wsb, torch.cuda.current_stream().cuda_stream)
    return [o.long().cpu() for o in outs]


def _scan(xyz, new_xyz, radii, ks):
    """psg_ball_query, the exhaustive scan."""
    from pointsecguard_b200 import _lib as L
    xyz, new_xyz = xyz.cuda().contiguous(), new_xyz.cuda().contiguous()
    nc, N, _ = xyz.shape
    P, S, _ = new_xyz.shape
    nr, r, k = _c_args(radii, ks)
    outs = [torch.full((P, S, kk), -7, dtype=torch.int32, device="cuda") for kk in ks]
    L.psg_ball_query(xyz.data_ptr(), nc, P, N, new_xyz.data_ptr(), S, nr, r, k, outs[0].data_ptr(),
                     outs[1].data_ptr() if nr == 2 else None, torch.cuda.current_stream().cuda_stream)
    return [o.long().cpu() for o in outs]


def _oracle(xyz, new_xyz, radii, ks):
    P = new_xyz.shape[0]
    clouds = xyz[torch.arange(P) % xyz.shape[0]]
    return [G.ball_query(r, k, clouds, new_xyz) for r, k in zip(radii, ks)]


def _check_ball(xyz, new_xyz, radii, ks, public=False):
    """grid == scan == oracle for every radius; the message counts the centroids whose index rows differ."""
    ref = _oracle(xyz, new_xyz, radii, ks)
    got = {"grid": _grid(xyz, new_xyz, radii, ks), "scan": _scan(xyz, new_xyz, radii, ks)}
    if public:
        assert xyz.shape[0] == new_xyz.shape[0]
        xd, qd = xyz.cuda(), new_xyz.cuda()
        if len(radii) == 1:
            got["op"] = [_psg().ball_query(radii[0], ks[0], xd, qd).cpu()]
        else:
            got["op"] = [t.cpu() for t in _psg().ball_query2(radii[0], ks[0], radii[1], ks[1], xd, qd)]
    bad = {}
    for path, outs in got.items():
        for r, k, o, e in zip(radii, ks, outs, ref):
            rows = int((o != e).any(-1).sum())
            if rows:
                bad[f"{path} r={r} K={k}"] = f"{rows} of {o.shape[0] * o.shape[1]} centroids"
    assert not bad, bad


# ---- ball query -----------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("radii", RADIUS_SETS, ids=["r" + "_".join(f"{r:g}" for r in rs) for rs in RADIUS_SETS])
@pytest.mark.parametrize("off", [t[0] for t in TRANSFORMS[:-2]], ids=TF_IDS[:-2])
def test_ball_query_translated(off, radii):
    xyz = _block(2, 4096, 1, off)
    new_xyz = _pick(xyz, 1024, 1)
    for ks in ([16], [32]) if len(radii) == 1 else ([32, 16], [16, 32]):
        _check_ball(xyz, new_xyz, radii, ks)


@gpu
@pytest.mark.parametrize("K", [1, 64, 128])
@pytest.mark.parametrize("offset", OFFSETS)
def test_public_op_translated(offset, K):
    """torch.ops.psg.ball_query / ball_query2 (the grid for N >= 1024) at the nsample edges."""
    xyz = _block(2, 4096, 2, (offset, offset, 0.0))
    new_xyz = _pick(xyz, 512, 2)
    _check_ball(xyz, new_xyz, (0.2,), (K,), public=True)
    _check_ball(xyz, new_xyz, (0.1, 0.4), (K, K), public=True)


@gpu
@pytest.mark.parametrize("radii", RADIUS_SETS[:5] + [(0.1, 0.05)], ids=lambda rs: "r" + "_".join(f"{r:g}" for r in rs))
@pytest.mark.parametrize("scale", [1e-3, 1e3], ids=["mm", "km"])
def test_ball_query_scaled(scale, radii):
    """Millimetre and kilometre clouds with the radii scaled alike (at 1e-3 the cell's 1e-4 term dominates)."""
    xyz = _block(2, 4096, 3, scale=scale)
    new_xyz = _pick(xyz, 1024, 3)
    rs = tuple(r * scale for r in radii)
    _check_ball(xyz, new_xyz, rs, (32,) * len(rs), public=True)


@gpu
def test_ball_query_scene_slab_with_dense_patch():
    """A 60 x 60 x 3 m slab of 65 536 points: far more than kMaxCells cells of 1.01 r, so the cell grows in x1.26 steps
    to several times r.  A dense patch of 1500 points in a 0.15 m cube puts 256 centroids above the 96-hit list: they
    take the exhaustive fallback while the others stay on the grid."""
    g = torch.Generator().manual_seed(5)
    N, S = 65536, 2048
    xyz = torch.rand(1, N, 3, generator=g) * torch.tensor([60.0, 60.0, 3.0]) - torch.tensor([30.0, 30.0, 0.0])
    patch = torch.randperm(N, generator=g)[:1500]
    xyz[0, patch] = torch.rand(1500, 3, generator=g) * 0.15 + torch.tensor([3.0, 4.0, 1.5])
    sel = torch.cat([patch[:256], torch.randperm(N, generator=g)[: S - 256]])
    new_xyz = xyz[:, sel].contiguous()
    _check_ball(xyz, new_xyz, (0.1,), (32,), public=True)
    _check_ball(xyz, new_xyz, (0.05, 0.1), (16, 32))


def _seam_cloud(counts, r_units=8, unit=1.0 / 64):
    """Centroids with exactly `counts[i]` hits at radius r_units * unit, every coordinate on a 2^-6 lattice and below
    8 m so that every distance is exact in fp32.  Each centroid gets two hits at exactly d2 = r^2 and all of its other
    lattice neighbours are placed just outside (d2 = r^2 + unit^2) or far away."""
    rng = np.random.default_rng(sum(counts))
    R = r_units
    v = np.stack(np.meshgrid(*[np.arange(-R, R + 1)] * 3, indexing="ij"), -1).reshape(-1, 3)
    n2 = (v ** 2).sum(1)
    inside, ring = v[(n2 <= R * R) & (n2 > 0)], v[n2 == R * R + 1]
    on_edge = np.array([[R, 0, 0], [0, -R, 0]])
    pts, cents = [], []
    for i, n in enumerate(counts):
        c = np.array([32 + 128 * i, 32, 64])                              # (0.5 + 2 i, 0.5, 1.0) m in lattice units
        rest = inside[~((inside[:, None] == on_edge[None]).all(-1).any(1))]
        own = np.concatenate([[[0, 0, 0]], on_edge, rest[rng.choice(len(rest), n - 3, replace=False)]])
        pts += [c + own, c + ring[rng.choice(len(ring), 20, replace=False)]]
        cents.append(c)
    far = rng.integers(0, 320, (1000, 3)) * np.array([1, 1, 0]) + np.array([0, 0, 256])   # a sheet 3 m above them
    pts.append(far)
    pts = np.concatenate(pts)
    pts = pts[rng.permutation(len(pts))]                                   # hits spread over the index range
    xyz = torch.from_numpy((pts * unit).astype(np.float32))[None]
    new_xyz = torch.from_numpy((np.array(cents) * unit).astype(np.float32))[None]
    return xyz, new_xyz


@gpu
@pytest.mark.parametrize("K", [32, 96, 128])
def test_ball_query_fallback_seam(K):
    """Exactly 95, 96, 97 and 98 hits (the grid keeps 96 per warp and falls back above), points at exactly d2 = r^2."""
    xyz, new_xyz = _seam_cloud([95, 96, 97, 98])
    r = 8.0 / 64
    ref = G.ball_query(r, 128, xyz, new_xyz)[0]
    for s, n in enumerate([95, 96, 97, 98]):                                 # the construction itself
        assert len(set(ref[s].tolist())) == n and ref[s, n - 1] > ref[s, 0]
    _check_ball(xyz, new_xyz, (r,), (K,))
    _check_ball(xyz, new_xyz, (r, r / 2), (K, K))
    _check_ball(xyz, new_xyz, (r / 2, r), (K, K))


def _cell(rmax):
    """grid_build_kernel's first cell edge, in float32."""
    return np.float32(np.float32(np.float32(rmax) * np.float32(1.01)) + np.float32(1e-4))


@gpu
@pytest.mark.parametrize("r", [0.1, 0.2])
def test_ball_query_points_on_cell_boundaries(r):
    """Coordinates exactly on cell boundaries (min + m * cell), one ulp either side of them, and centroids there."""
    cell = _cell(r)
    xyz = _block(1, 2048, 7)
    xyz[0, 0] = torch.tensor([-0.5, -0.5, 0.0])                               # pins the bounding box's minimum
    xyz[0, 1] = torch.tensor([0.5, 0.5, 3.0])
    g = torch.Generator().manual_seed(8)
    lo = np.array([-0.5, -0.5, 0.0], np.float32)
    for a in range(3):
        m = torch.randint(1, int(np.floor((3.0 if a == 2 else 1.0) / cell)), (600,), generator=g).numpy()
        b = (lo[a] + m.astype(np.float32) * cell).astype(np.float32)
        b = np.where(np.arange(600) % 3 == 1, np.nextafter(b, np.float32(np.inf)), b)
        b = np.where(np.arange(600) % 3 == 2, np.nextafter(b, np.float32(-np.inf)), b)
        rows = torch.randperm(2046, generator=g)[:600] + 2
        xyz[0, rows, a] = torch.from_numpy(b.astype(np.float32))
    new_xyz = _pick(xyz, 512, 9)
    _check_ball(xyz, new_xyz, (r,), (32,), public=True)
    _check_ball(xyz, new_xyz, (r, r / 2), (32, 16))


@gpu
@pytest.mark.parametrize("offset", [0.0, 100.0])
def test_ball_query_shared_clouds_and_free_centroids(offset):
    """nclouds < P (three problems per cloud) and centroids that are not cloud points: inside the bounding box, just
    outside it and far outside it."""
    nc, P, N, S = 2, 6, 4096, 256
    xyz = _block(nc, N, 11, (offset, offset, 0.0))
    g = torch.Generator().manual_seed(12)
    q = torch.rand(P, S, 3, generator=g)
    q[..., :2] = q[..., :2] * 1.4 - 0.7                                        # 0.2 m beyond the box in x and y
    q[..., 2] = q[..., 2] * 3.6 - 0.3
    q[:, :16] += torch.tensor([3.0, -4.0, 5.0])                               # far outside
    new_xyz = (q + torch.tensor([offset, offset, 0.0])).contiguous()
    for radii, ks in (((0.1,), (32,)), ((0.4,), (16,)), ((0.2, 0.1), (32, 16))):
        _check_ball(xyz, new_xyz, radii, ks)


@gpu
@pytest.mark.parametrize("N", [1, 3, 31, 33, 1023, 1024, 2047, 2048])
def test_ball_query_cloud_sizes(N):
    """Around the public op's scan / grid switch (N = 1024) and the engine's (N = 2048)."""
    xyz = _block(2, N, 13)
    g = torch.Generator().manual_seed(14)
    new_xyz = (torch.rand(2, 40, 3, generator=g) * torch.tensor([1.0, 1.0, 3.0]) - torch.tensor([0.5, 0.5, 0.0]))
    new_xyz = torch.cat([new_xyz, xyz[:, : min(N, 24)]], 1).contiguous()
    _check_ball(xyz, new_xyz, (0.2,), (16,), public=True)
    _check_ball(xyz, new_xyz, (0.8, 0.4), (32, 16), public=True)


# ---- 3-NN -----------------------------------------------------------------------------------------------------------
@pytest.fixture
def nn_grid():
    """Sets the 3-NN kernel choice (1: exhaustive kernel, 2: grid whenever S fits) and restores automatic choice."""
    from pointsecguard_b200 import _lib as L
    yield lambda m: L.psg_set_option(b"nn_grid", m)
    L.psg_set_option(b"nn_grid", 0)


def _nn_equal(a, b):
    return a.shape == b.shape and bool(torch.equal(torch.isnan(a), torch.isnan(b))) and \
        bool(torch.equal(torch.nan_to_num(a, nan=0.0), torch.nan_to_num(b, nan=0.0)))


def _check_three_nn(nn_grid, xyz1, xyz2):
    ref = G.three_nn(xyz1, xyz2)
    bad = []
    for mode in (1, 2):
        nn_grid(mode)
        got = [t.cpu() for t in _psg().three_nn(xyz1.cuda(), xyz2.cuda())]
        for name, o, e in zip(("idx", "d2", "w"), got, ref):
            if not _nn_equal(o, e):
                bad.append(f"mode {mode} {name}: {int((o != e).any(-1).sum())} rows differ")
    assert not bad, bad


@gpu
@pytest.mark.parametrize("S", [3, 255, 256, 2048, 2049])
@pytest.mark.parametrize("tf", TRANSFORMS, ids=TF_IDS)
def test_three_nn_translated_and_scaled(nn_grid, tf, S):
    """Every cloud point queries an S-point subset of its own cloud, so every candidate is also a query at d = 0 (its
    weight normalises 1e8 terms).  S covers the grid's automatic choice (256) and its limit kNgMaxS = 2048."""
    off, scale = tf
    xyz = _block(2, 4096, 21, off, scale)
    _check_three_nn(nn_grid, xyz, _pick(xyz, S, 22))


# ---- FPS and square_distance ----------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("N,S", [(4096, 1024), (20000, 256)])
@pytest.mark.parametrize("tf", TRANSFORMS, ids=TF_IDS)
def test_fps_and_square_distance_translated_and_scaled(tf, N, S):
    off, scale = tf
    xyz = _block(2, N, 31, off, scale)
    start = torch.randint(0, N, (2,), generator=torch.Generator().manual_seed(32))
    assert torch.equal(_psg().fps(xyz.cuda(), S, start).cpu(), G.fps(xyz, S, start))
    src = _pick(xyz, 256, 33)
    dst = xyz[:, :2048].contiguous()
    assert torch.equal(_psg().square_distance(src.cuda(), dst.cuda()).cpu(), G.square_distance(src, dst))


# ---- the engine -----------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("N", [2047, 2048, 4096])
def test_engine_indices_on_a_translated_block(N):
    """The SSG engine's resident index buffers on a painted block moved 100 m in x and y.  N >= 2048 bins SA1 through
    the ball grid (N = 4096 is the benchmark's size); 2047 is the last scan."""
    from pointsecguard_b200.models.pointnet2_sem_seg import get_model
    m = get_model(13)
    m.load_state_dict(syn.load_checkpoint("ssg"))
    m = m.cuda().eval()
    x, _ = syn.make_painted_blocks(1, N, 3)
    x[:, 0:2] += 100.0
    eng = m.engine(torch.device("cuda"))
    eng.bind(1, N, 1)
    eng.set_input(x.cuda())
    torch.manual_seed(7)
    starts = eng.draw_starts(1)
    eng.geometry(starts)
    clouds = [x[:, :3].permute(0, 2, 1).contiguous()]
    for l, (S, r, K) in enumerate([(1024, 0.1, 32), (256, 0.2, 32), (64, 0.4, 32), (16, 0.8, 32)], start=1):
        fps = G.fps(clouds[-1], S, starts[l - 1, 0].long())
        assert np.array_equal(eng.read_geometry("fps", l).cpu().numpy(), fps.numpy().astype(np.int32)), ("fps", l)
        new_xyz = torch.gather(clouds[-1], 1, fps.unsqueeze(-1).expand(-1, -1, 3))
        assert torch.equal(eng.read_geometry("xyz", l).cpu(), new_xyz), ("xyz", l)
        ball = G.ball_query(r, K, clouds[-1], new_xyz).numpy().astype(np.int32)
        got = eng.read_geometry("ball", l).cpu().numpy()
        assert np.array_equal(got, ball), ("ball", l, int((got != ball).any(-1).sum()), "centroids differ")
        clouds.append(new_xyz)
    for f in range(4):
        idx, d2, w = G.three_nn(clouds[f], clouds[f + 1])
        assert np.array_equal(eng.read_geometry("nn_idx", f).cpu().numpy(), idx.numpy().astype(np.int32)), ("nn", f)
        assert torch.equal(eng.read_geometry("nn_w", f).cpu(), w), ("nn_w", f)


# ---- non-finite coordinates -----------------------------------------------------------------------------------------
@gpu
def test_ball_query_nan_counts_as_the_reference_counts_it():
    """A NaN distance is a hit (pointnet_util.py:102 keeps what is not > r^2): a NaN point is in every centroid's ball,
    a NaN centroid takes the first K points.  The grid must agree with the scan and the oracle."""
    xyz = _block(2, 4096, 41)
    new_xyz = _pick(xyz, 256, 41)
    xyz[0, 100, 0] = float("nan")
    xyz[0, 3000] = float("nan")
    xyz[1, 7, 2] = float("nan")
    new_xyz[0, 5] = float("nan")
    new_xyz[1, 9, 1] = float("nan")
    _check_ball(xyz, new_xyz, (0.1,), (32,), public=True)
    _check_ball(xyz, new_xyz, (0.2, 0.1), (32, 16), public=True)


@gpu
def test_ball_query_infinite_coordinates():
    """A cloud with infinite coordinates is not binned: every centroid takes the scan, so the grid returns what the
    scan and the oracle return (the distance formula's inf - inf = NaN counts as a hit)."""
    xyz = _block(1, 4096, 42)
    new_xyz = _pick(xyz, 256, 42)
    xyz[0, 10, 0] = float("inf")
    xyz[0, 20, 2] = float("-inf")
    new_xyz[0, 3, 1] = float("inf")
    _check_ball(xyz, new_xyz, (0.1,), (32,), public=True)


@gpu
@pytest.mark.parametrize("S", [256, 2048])
def test_three_nn_non_finite(nn_grid, S):
    """NaN and infinite queries and candidates: the grid kernel scans such queries in index order, so it returns what
    the exhaustive kernel and the oracle return (NaN weights included)."""
    xyz = _block(2, 4096, 43)
    xyz2 = _pick(xyz, S, 44)
    xyz[0, 5, 0] = float("nan")
    xyz[0, 6] = float("inf")
    xyz[1, 9, 2] = float("-inf")
    xyz2[1, 17, 1] = float("nan")
    _check_three_nn(nn_grid, xyz, xyz2)
    xyz2[1, 17, 1] = float("inf")
    _check_three_nn(nn_grid, xyz, xyz2)


# ---- CPU: why the ball grid needs its margin rule -------------------------------------------------------------------
def _grid_cells(xyz, rmax, max_cells=16384):
    """grid_build_kernel's cell assignment in float32: bounding box, cell = 1.01 r + 1e-4 grown x1.26 until the grid
    has at most kMaxCells cells, floor((x - min) / cell) clamped to the grid.  Returns (cells [N, 3], cell, max |p|^2)."""
    lo, hi = xyz.min(0), xyz.max(0)
    cell = _cell(rmax)
    while True:
        g = np.floor((hi - lo) / cell) + 1
        if np.prod(g.astype(np.float64)) <= max_cells:
            break
        cell = np.float32(cell * np.float32(1.26))
    inv = np.float32(np.float32(1.0) / cell)
    c = np.floor((xyz - lo) * inv).astype(np.int64)
    return np.clip(c, 0, g.astype(np.int64) - 1).astype(np.int32), cell, _sqnorm(xyz).max()


def _sqnorm(p):
    return (p[..., 0] * p[..., 0] + p[..., 1] * p[..., 1]) + p[..., 2] * p[..., 2]


def _grid_serves(qn, m2, cell, r):
    """ball_grid_kernel's margin rule: 2^-19 (|q|^2 + max|p|^2 + cell^2) < cell^2 - r^2."""
    c2 = np.float32(cell * cell)
    return np.float32(2.0 ** -19) * ((qn + m2) + c2) < c2 - np.float32(r * r)


def _hits_outside_visited_cells(offset, r, N=4096, S=1024, seed=0):
    """Oracle hits (every hit: nsample = N) that lie outside the 27 cells the grid visits, per centroid."""
    xyz = _block(1, N, seed, (offset, offset, 0.0))
    sel = torch.randperm(N, generator=torch.Generator().manual_seed(seed + 1))[:S]
    q = xyz[:, sel]
    ref = G.ball_query(r, N, xyz, q)[0].numpy()
    x = xyz[0].numpy()
    cells, cell, m2 = _grid_cells(x, r)
    cq = cells[sel.numpy()]
    real = np.ones_like(ref, bool)
    real[:, 1:] = ref[:, 1:] != ref[:, :1]                                  # padding repeats the first hit
    real &= ref < N
    far = (np.abs(cells[np.minimum(ref, N - 1)] - cq[:, None]) > 1).any(-1) & real
    return far.sum(1), _grid_serves(_sqnorm(q[0].numpy()), m2, cell, r)


def test_ball_grid_margin_rule_covers_translated_clouds():
    """At 100 m from the origin the 27 visited cells miss oracle hits (the expansion formula's error, ~2^-24 |p|^2,
    exceeds the cell margin cell^2 - r^2), and the margin rule sends every such centroid to the exhaustive scan.  At
    the origin nothing is missed and the rule keeps the grid for every centroid, at r = 0.1 and at 0.05."""
    for r in (0.1, 0.05):
        missed, serves = _hits_outside_visited_cells(0.0, r)
        assert missed.sum() == 0 and serves.all(), r
    missed, serves = _hits_outside_visited_cells(100.0, 0.1)
    assert missed.sum() > 0
    assert not serves[missed > 0].any()
