"""The training kernels of csrc/train.cu one by one through the C ABI, against fp64 references computed on the CPU from
the same fp32 inputs, at the row counts that hit their tile and split edges.

T-layout buffers are built and read here directly in torch (float T[rows/128][wchunks][128][4]), not by the pack kernels.
Every padded row and column of every input view is NaN, so a kernel that reads past the real data yields a non-finite
output.  Each gate is an error bound in units of u = 2^-24 times the magnitudes involved; the tests print the measured
max err / bound.  The reductions also run a control: the same reference with the rows of the final 128-row tile left out
(or with the bug class named) must miss the gate by at least 10x, so the gate is sharp enough to see that tile.
"""
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

U = 2.0 ** -24
NAN = float("nan")
# rows: 1 tile / 1 split; first partial tile; two tiles; 8 tiles (BN 4 splits of 2, wgrad 8 of 1); 594 tiles (C = 4:
# 297 splits of 2; C = 64: 35 splits, the last of 16 tiles, the last tile partial); 1002 tiles (wgrad one output tile:
# 501 splits of 2); B = 16 SA1 training rows
EDGE_ROWS = [1, 2, 127, 128, 129, 1000, 128 * 593 + 5, 128 * 1001 + 77]
BIG_ROWS = 524288


def _L():
    from pointsecguard_b200 import _lib as L
    return L


def _st():
    return torch.cuda.current_stream().cuda_stream


def to_t(x, wchunks=None, c0=0, fill=NAN):
    """x [rows, C] -> T-layout buffer (flat, CUDA) with the columns at chunk c0 of a view `wchunks` wide; everything else
    (padded rows, other columns) = fill"""
    rows, C = x.shape
    if wchunks is None:
        wchunks = (C + 15) // 16 * 4
    rpad = (rows + 127) // 128 * 128
    full = torch.full((rpad, wchunks * 4), fill, dtype=torch.float32)
    full[:rows, 4 * c0: 4 * c0 + C] = x.float().cpu()
    return full.view(rpad // 128, 128, wchunks, 4).permute(0, 2, 1, 3).contiguous().view(-1).cuda()


def from_t(buf, rows, wchunks):
    """T-layout buffer -> [rpad, 4 * wchunks] on the CPU (padded rows included)"""
    rpad = buf.numel() // (4 * wchunks)
    return buf.cpu().view(rpad // 128, wchunks, 128, 4).permute(0, 2, 1, 3).reshape(rpad, 4 * wchunks)


def ulp(x):
    """spacing of float32 at |x| (x fp64 tensor)"""
    return torch.from_numpy(np.spacing(np.abs(x.numpy()).astype(np.float32)).astype(np.float64))


def ratio(got, ref, bound):
    """max |got - ref| / bound (fp64), got must be finite"""
    got = got.double()
    assert torch.isfinite(got).all()
    return ((got - ref).abs() / bound).max().item()


def _wchunks(C):
    return (C + 15) // 16 * 4


def _gen(seed):
    return torch.Generator().manual_seed(seed)


# ----------------------------------------------------------------------------------------------------------------------
# BatchNorm forward
# ----------------------------------------------------------------------------------------------------------------------
def _bn_cases():
    out = []
    for rows in EDGE_ROWS:
        for C in (4, 20, 64):
            out.append((rows, C))
    out += [(1000, 128), (129, 1024), (128 * 593 + 5, 128), (2000, 1024), (BIG_ROWS, 32), (BIG_ROWS, 64)]
    return out


BN_CASES = _bn_cases()


def _bn_forward(z, C, gamma, beta, rm, rv, mom, eps, relu, wz=None):
    L = _L()
    rows = z.shape[0]
    wz = wz or _wchunks(C)
    zt = to_t(z, wz)
    yt = torch.full_like(zt, NAN)
    sm = torch.full((C,), NAN, device="cuda")
    si = torch.full((C,), NAN, device="cuda")
    ws = torch.empty(L.psg_bn_workspace(C), dtype=torch.uint8, device="cuda")
    rmd = rm.clone().cuda() if rm is not None else None
    rvd = rv.clone().cuda() if rv is not None else None
    gd, bd = gamma.cuda(), beta.cuda()                               # (kept alive until the kernels have run)
    L.psg_bn_train_forward(zt.data_ptr(), wz, rows, C, gd.data_ptr(), bd.data_ptr(),
                           rmd.data_ptr() if rmd is not None else None, rvd.data_ptr() if rvd is not None else None,
                           mom, eps, yt.data_ptr(), wz, relu, sm.data_ptr(), si.data_ptr(), ws.data_ptr(), ws.numel(), _st())
    torch.cuda.synchronize()
    return from_t(yt, rows, wz), sm.cpu(), si.cpu(), (rmd.cpu() if rmd is not None else None), (rvd.cpu() if rvd is not None else None)


def _bn_inputs(rows, C, seed, offset):
    g = _gen(seed)
    z = torch.randn(rows, C, generator=g) * (0.5 + torch.rand(C, generator=g)) + offset
    z[:, C // 2] = 0.37                           # a constant column: var = 0 -> invstd = 1 / sqrt(eps)
    gamma = 0.5 + torch.rand(C, generator=g)
    beta = torch.randn(C, generator=g)
    rm = torch.randn(C, generator=g)
    rv = 0.5 + torch.rand(C, generator=g)
    return z, gamma, beta, rm, rv


@pytest.mark.parametrize("offset", [0.0, 1000.0], ids=["randn", "offset1000"])
@pytest.mark.parametrize("case", BN_CASES, ids=[f"{r}x{c}" for r, c in BN_CASES])
def test_bn_forward(case, offset):
    rows, C = case
    if offset and rows > 200000 and C > 32:
        pytest.skip("one large offset case is enough")
    z, gamma, beta, rm, rv = _bn_inputs(rows, C, rows * 7 + C, offset)
    relu = (rows + C) % 2
    mom = 0.1 if C % 8 else 0.3
    track = rows % 3 != 2
    eps = 1e-5
    y, sm, si, rm1, rv1 = _bn_forward(z, C, gamma, beta, rm if track else None, rv if track else None, mom, eps, relu)
    zd = z.double()
    mean = zd.mean(0)
    var = ((zd - mean) ** 2).mean(0)                                  # two-pass, biased
    eps32 = float(np.float32(eps))
    invstd = 1.0 / torch.sqrt(var + eps32)
    r_mean = ratio(sm, mean, 4 * ulp(mean) + 1e-300)
    r_inv = ratio(si, invstd, 4 * ulp(invstd))
    # y = relu?(z * alpha + beta') in fp32 from the saved statistics: alpha, mean * alpha, the difference and the fma each
    # round once -> 4u (|z alpha| + |beta| + |mean alpha|), |beta'| <= |beta| + |mean alpha|
    alpha = si.double() * gamma.double()
    bp = beta.double() - sm.double() * alpha
    yref = zd * alpha + bp
    if relu:
        yref = yref.clamp_min(0)
    ybound = 4 * U * (zd.abs() * alpha.abs() + beta.double().abs() + (sm.double() * alpha).abs()) + 1e-300
    r_y = ratio(y[:rows, :C], yref, ybound)
    assert (y[rows:, :C] == 0).all(), "rows past the end of y must be zero"
    msg = f"bn fwd {rows}x{C} off {offset}: mean {r_mean:.3f} invstd {r_inv:.3f} y {r_y:.3f}"
    worst = max(r_mean, r_inv, r_y)
    if track:
        m32 = float(np.float32(mom))                                 # the kernel promotes the fp32 momentum
        unb = rows / (rows - 1) if rows > 1 else 1.0
        rm_ref = (1 - m32) * rm.double() + m32 * mean
        rv_ref = (1 - m32) * rv.double() + m32 * var * unb
        rv_bound = 2 * ulp(rv_ref)
        r_rm = ratio(rm1, rm_ref, 2 * ulp(rm_ref) + 1e-300)
        r_rv = ratio(rv1, rv_ref, rv_bound)
        worst = max(worst, r_rm, r_rv)
        msg += f" running mean {r_rm:.3f} var {r_rv:.3f}"
        if 1 < rows <= 2000 and offset == 0:
            # control: the biased variance in the running update
            ctl = ratio(rv1, (1 - m32) * rv.double() + m32 * var, rv_bound)
            msg += f" | control biased var {ctl:.1f}"
            assert ctl >= 10
    print(msg)
    assert worst < 1, msg


def test_bn_forward_matches_torch_batchnorm():
    """The momentum / unbiased-variance semantics pinned against torch.nn.BatchNorm1d itself."""
    rows, C = 1000, 64
    z, gamma, beta, rm, rv = _bn_inputs(rows, C, 5, 0.0)
    bn = torch.nn.BatchNorm1d(C, momentum=0.3).cuda().train()
    with torch.no_grad():
        bn.weight.copy_(gamma)
        bn.bias.copy_(beta)
        bn.running_mean.copy_(rm)
        bn.running_var.copy_(rv)
        yt = torch.relu(bn(z.cuda())).cpu()
    y, sm, si, rm1, rv1 = _bn_forward(z, C, gamma, beta, rm, rv, 0.3, bn.eps, 1)
    # torch's own float arithmetic differs; 1e-5 relative is far below the biased / unbiased difference (1e-4 * 0.3 var)
    # and any momentum mix-up
    assert torch.allclose(rm1, bn.running_mean.cpu(), rtol=1e-5, atol=1e-6)
    assert torch.allclose(rv1, bn.running_var.cpu(), rtol=1e-5, atol=1e-6)
    assert torch.allclose(y[:rows, :C], yt, rtol=1e-4, atol=1e-5)


# ----------------------------------------------------------------------------------------------------------------------
# BatchNorm backward
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("alias", [0, 1], ids=["dz", "dz_is_dy"])
@pytest.mark.parametrize("with_y", [0, 1], ids=["noy", "relu"])
@pytest.mark.parametrize("case", BN_CASES, ids=[f"{r}x{c}" for r, c in BN_CASES])
def test_bn_backward(case, with_y, alias):
    L = _L()
    rows, C = case
    if rows * C > 4_000_000 and (with_y, alias) != (1, 1):
        pytest.skip("the large cases run as train.py calls them (ReLU, dz aliasing dy)")
    g = _gen(rows * 3 + C)
    w = _wchunks(C)
    z = torch.randn(rows, C, generator=g) * 2 + 0.3
    dy = 1.0 + torch.randn(rows, C, generator=g)                    # non-zero mean: dbeta / n is O(1)
    y = torch.relu(torch.randn(rows, C, generator=g)) if with_y else None
    gamma = 0.5 + torch.rand(C, generator=g)
    mu = torch.randn(C, generator=g) * 0.1 + 0.3
    inv = 0.4 + torch.rand(C, generator=g)
    dyt, zt = to_t(dy, w), to_t(z, w)
    yt = to_t(y, w) if with_y else None
    dzt = dyt if alias else torch.full_like(dyt, NAN)
    dgam = torch.full((C,), NAN, device="cuda")
    dbet = torch.full((C,), NAN, device="cuda")
    ws = torch.empty(L.psg_bn_workspace(C), dtype=torch.uint8, device="cuda")
    gmd, mud, ivd = gamma.cuda(), mu.cuda(), inv.cuda()
    L.psg_bn_train_backward(dyt.data_ptr(), w, yt.data_ptr() if with_y else None, w if with_y else 0, zt.data_ptr(), w,
                            rows, C, gmd.data_ptr(), mud.data_ptr(), ivd.data_ptr(), dgam.data_ptr(),
                            dbet.data_ptr(), dzt.data_ptr(), w, ws.data_ptr(), ws.numel(), _st())
    torch.cuda.synchronize()
    dz = from_t(dzt, rows, w)
    assert (dz[rows:, :C] == 0).all(), "rows past the end of dz must be zero"
    gd = dy.double() * (y.double() > 0) if with_y else dy.double()
    xh = (z.double() - mu.double()) * inv.double()
    db_ref = gd.sum(0)
    dg_ref = (gd * xh).sum(0)
    r_db = ratio(dbet.cpu(), db_ref, ulp(db_ref) + 1e-300)
    dg_bound = 4 * U * (gd * xh).abs().sum(0) + 1e-300
    r_dg = ratio(dgam.cpu(), dg_ref, dg_bound)
    gi = gamma.double() * inv.double()

    def dz_of(gg, n, dbr, dgr):
        return (gg - dbr / n - xh * dgr / n) * gi

    # each term of (g - dbeta/n - xhat dgamma/n) gamma invstd carries at most ~10 fp32 roundings; plus the dgamma error
    dz_bound = (10 * U * gi.abs() * (gd.abs() + db_ref.abs() / rows + (xh * dg_ref).abs() / rows)
                + gi.abs() * xh.abs() * dg_bound / rows + 1e-300)
    r_dz = ratio(dz[:rows, :C], dz_of(gd, rows, db_ref, dg_ref), dz_bound)
    msg = f"bn bwd {rows}x{C} y {with_y} alias {alias}: dbeta {r_db:.3f} dgamma {r_dg:.3f} dz {r_dz:.3f}"
    if with_y:   # control: the ReLU mask ignored
        ctl = ratio(dz[:rows, :C], dz_of(dy.double(), rows, dy.double().sum(0), (dy.double() * xh).sum(0)), dz_bound)
        msg += f" | control no mask {ctl:.1f}"
        assert ctl >= 10
    if 1 < rows <= 200000:   # control: n off by one (visible where g = 0 and dbeta / n is O(1))
        ctl = ratio(dz[:rows, :C], dz_of(gd, rows - 1, db_ref, dg_ref), dz_bound)
        msg += f" n-1 {ctl:.1f}"
        assert ctl >= 10
    print(msg)
    assert max(r_db, r_dg, r_dz) < 1, msg


# ----------------------------------------------------------------------------------------------------------------------
# weight gradient
# ----------------------------------------------------------------------------------------------------------------------
# (rows, cout, k1, k2, a1 view (wchunks, c0), a2 view (wchunks, c0), dz wchunks)
def _wg_cases():
    out = []
    for rows in EDGE_ROWS:
        out.append((rows, 13, 13, 0, None, None, None))
        out.append((rows, 32, 12, 0, None, None, None))                  # SA1 first layer
    out += [
        (BIG_ROWS, 32, 12, 0, None, None, None),
        (65536, 256, 64, 256, None, None, None), (1000, 256, 256, 512, None, None, None),     # FP two-source
        (128 * 593 + 5, 13, 128, 0, None, None, None), (129, 13, 128, 0, None, None, None),   # head conv2
        (1000, 1, 1, 0, None, None, None), (128 * 1001 + 77, 65, 13, 0, None, None, None), (127, 65, 1, 0, None, None, None),
        (1000, 13, 20, 12, (12, 2), (8, 3), None), (128 * 593 + 5, 65, 20, 13, (8, 1), (8, 4), None),
        (129, 40, 20, 12, None, None, 16),                                # dz view wider than cout
    ]
    return out


WG_CASES = _wg_cases()


def _wg_id(c):
    rows, cout, k1, k2, v1, v2, wd = c
    return f"{rows}r_{cout}x{k1}+{k2}" + ("_views" if v1 else "") + ("_wide" if wd else "")


@pytest.mark.parametrize("acc", [0, 1], ids=["set", "acc"])
@pytest.mark.parametrize("case", WG_CASES, ids=[_wg_id(c) for c in WG_CASES])
def test_conv_wgrad(case, acc):
    L = _L()
    rows, cout, k1, k2, v1, v2, wdz = case
    g = _gen(rows + cout * 7 + k1 * 31 + k2)
    dz = torch.randn(rows, cout, generator=g)
    if rows > 1:
        dz -= dz.mean(0)                                               # zero-mean columns, as BatchNorm's backward makes
    a1 = torch.randn(rows, k1, generator=g) + 0.5
    a2 = torch.randn(rows, k2, generator=g) - 0.25 if k2 else None
    w1, c1 = v1 or (_wchunks(k1), 0)
    w2, c2 = v2 or ((_wchunks(k2), 0) if k2 else (0, 0))
    wz = wdz or _wchunks(cout)
    dzt, a1t = to_t(dz, wz), to_t(a1, w1, c1)
    a2t = to_t(a2, w2, c2) if k2 else None
    cin = k1 + k2
    pre = torch.randn(cout, cin, generator=g)
    dW = pre.clone().cuda() if acc else torch.full((cout, cin), NAN, device="cuda")
    with_db = (rows + acc) % 2 == 1 or cout == 13
    db = torch.full((cout,), NAN, device="cuda") if with_db else None
    ws = torch.empty(L.psg_wgrad_workspace(cout, cin, rows), dtype=torch.uint8, device="cuda")
    L.psg_conv_wgrad(dzt.data_ptr(), wz, cout, a1t.data_ptr(), w1, c1, k1, a2t.data_ptr() if k2 else None, w2, c2, k2, rows,
                     dW.data_ptr(), db.data_ptr() if with_db else None, acc, ws.data_ptr(), ws.numel(), _st())
    torch.cuda.synchronize()
    x = torch.cat([a1, a2], 1) if k2 else a1
    dzd, xd = dz.double(), x.double()
    ref = dzd.t() @ xd
    l2 = torch.sqrt((dzd ** 2).t() @ (xd ** 2))                      # || (dz_rn x_rk)_r ||_2
    bound = 16 * U * math.sqrt(rows) * l2 + 1e-300
    if acc:
        ref = ref + pre.double()
        bound = bound + U * ref.abs()
    r_w = ratio(dW.cpu(), ref, bound)
    msg = f"wgrad {_wg_id(case)} acc {acc}: dW {r_w:.3f}"
    if with_db:
        db_ref = dzd.sum(0)
        # overwritten, never accumulated; 1 ulp plus the double partial sums (zero-mean columns make db a sum that cancels)
        r_b = ratio(db.cpu(), db_ref, ulp(db_ref) + 2.0 ** -43 * dzd.abs().sum(0))
        msg += f" db {r_b:.3f}"
        r_w = max(r_w, r_b)
    # control: the final row tile dropped
    last = (rows - 1) // 128 * 128
    ctl_ref = dzd[:last].t() @ xd[:last] + (pre.double() if acc else 0)
    ctl = ratio(dW.cpu(), ctl_ref, bound)
    msg += f" | control last tile {ctl:.1f}"
    print(msg)
    assert r_w < 1, msg
    assert ctl >= 10, msg


# ----------------------------------------------------------------------------------------------------------------------
# head: log-softmax and its autograd
# ----------------------------------------------------------------------------------------------------------------------
HEAD_ROWS = [1, 255, 256, 257, 100003]


def _logits(rows, ncls, scale, seed):
    g = _gen(seed)
    z = torch.randn(rows, ncls, generator=g) if scale == 1 else torch.where(
        torch.rand(rows, ncls, generator=g) < 0.5, torch.tensor(-80.0), torch.tensor(80.0)) + torch.randn(rows, ncls, generator=g) * 0.01
    if rows >= 4:
        z[rows // 4] = 1.25                                            # a constant row
        z[rows // 2, :2] = z[rows // 2].max()                          # an exact tie for the maximum
    return z


@pytest.mark.parametrize("scale", [1, 80], ids=["unit", "pm80"])
@pytest.mark.parametrize("ncls", [2, 3, 4, 5, 8, 13, 16])
@pytest.mark.parametrize("rows", HEAD_ROWS)
def test_head_log_softmax_and_grad(rows, ncls, scale):
    L = _L()
    z = _logits(rows, ncls, scale, rows * 17 + ncls)
    zt = to_t(z, 4)
    logp = torch.full((rows, ncls), NAN, device="cuda")
    L.psg_log_softmax_rows(zt.data_ptr(), 4, rows, ncls, logp.data_ptr(), _st())
    dlogp = torch.randn(rows, ncls, generator=_gen(rows + ncls))
    dzt = torch.full_like(zt, NAN)
    dld = dlogp.cuda()
    L.psg_dlogits_from_dlogp(zt.data_ptr(), 4, dld.data_ptr(), rows, ncls, dzt.data_ptr(), 4, _st())
    torch.cuda.synchronize()
    zd = z.double()
    d = zd - zd.max(1, keepdim=True).values
    lref = torch.log_softmax(zd, 1)
    # (z - max) rounds once, exp 2 ulp, a recursive sum of ncls terms, log 1 ulp, the final difference once
    lbound = U * (4 * d.abs() + 4 * math.log(ncls) + ncls + 4)
    r_l = ratio(logp.cpu(), lref, lbound)
    p = torch.softmax(zd, 1)
    dd = dlogp.double()
    dref = dd - p * dd.sum(1, keepdim=True)
    # dz = dlogp - p * sum(dlogp): p carries the exp argument (u |z - max|), exp, the sum of ncls terms, 1 / s and one
    # product; the ncls-term sum of dlogp, the product p * s and the difference round once each
    dbound = U * (2 * dd.abs() + (2 * ncls + 12 + d.abs()) * p * dd.abs().sum(1, keepdim=True)) + 1e-300
    dz = from_t(dzt, rows, 4)
    r_d = ratio(dz[:rows, :ncls], dref, dbound)
    assert (dz[:rows, ncls:] == 0).all(), "columns ncls..15 of dz are written as zeros"
    print(f"head {rows}x{ncls} scale {scale}: logp {r_l:.3f} dz {r_d:.3f}")
    assert r_l < 1 and r_d < 1


@pytest.mark.parametrize("ncls", [1, 17])
def test_head_rejects_class_counts(ncls):
    L = _L()
    zt = torch.zeros(128 * 32, device="cuda")
    out = torch.zeros(128 * 32, device="cuda")
    with pytest.raises(L.PsgError):
        L.psg_log_softmax_rows(zt.data_ptr(), 8, 100, ncls, out.data_ptr(), _st())
    with pytest.raises(L.PsgError):
        L.psg_dlogits_from_dlogp(zt.data_ptr(), 8, out.data_ptr(), 100, ncls, out.data_ptr(), 8, _st())


# ----------------------------------------------------------------------------------------------------------------------
# weighted NLL
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("gout", [0, 1], ids=["g1", "g2.5"])
@pytest.mark.parametrize("weighted", [0, 1], ids=["now", "w"])
@pytest.mark.parametrize("ncls", [2, 13, 16, 40])
@pytest.mark.parametrize("rows", [1, 255, 256, 257, 262147, 1000000])
def test_nll_loss(rows, ncls, weighted, gout):
    L = _L()
    if rows == 1000000 and (weighted, gout) != (1, 1):
        pytest.skip("one large case per class count")
    g = _gen(rows + ncls * 3 + weighted)
    logp = torch.log_softmax(torch.randn(rows, ncls, generator=g) * 2, 1)
    lab = torch.randint(0, ncls, (rows,), generator=g)
    lab[torch.rand(rows, generator=g) < 0.05] = -100
    lab[0] = 0                                         # at least one counted row
    if rows > 2:
        lab[1] = ncls                                  # out of range above: ignored like -100
    w = (0.2 + torch.rand(ncls, generator=g)) if weighted else None
    out = torch.full((2,), NAN, device="cuda")
    ws = torch.empty(L.psg_nll_workspace(), dtype=torch.uint8, device="cuda")
    labd, logpd = lab.cuda(), logp.cuda()
    wd = w.cuda() if weighted else None
    L.psg_nll_loss(logpd.data_ptr(), labd.data_ptr(), wd.data_ptr() if weighted else None, rows, ncls, out.data_ptr(),
                   out[1:].data_ptr(), ws.data_ptr(), ws.numel(), _st())
    go = torch.tensor([2.5], device="cuda")
    dl = torch.full((rows, ncls), NAN, device="cuda")
    L.psg_nll_loss_backward(labd.data_ptr(), wd.data_ptr() if weighted else None, rows, ncls, go.data_ptr() if gout else None,
                            out[1:].data_ptr(), dl.data_ptr(), _st())
    torch.cuda.synchronize()
    # reference on the CPU (torch's CUDA nll_loss asserts on out-of-range labels)
    valid = (lab >= 0) & (lab < ncls)
    wv = (w.double()[lab[valid]] if weighted else torch.ones(int(valid.sum()), dtype=torch.float64))
    num = -(wv * logp.double()[valid.nonzero()[:, 0], lab[valid]]).sum()
    den = wv.sum()
    loss_ref, o = num / den, out.cpu()
    r_loss = abs(o[0].item() - loss_ref.item()) / (2 * ulp(loss_ref.reshape(1)).item())
    r_ws = abs(o[1].item() - den.item()) / (2 * ulp(den.reshape(1)).item())
    # backward: -w[y] * (1 / wsum) * g at the label, in fp32 exactly as the kernel orders it, and within the four roundings
    # (wsum, 1 / wsum and two products) of fp64
    gval = 2.5 if gout else 1.0
    inv = torch.tensor(1.0, dtype=torch.float32) / o[1]
    exp32 = torch.zeros(rows, ncls)
    wl = (w[lab[valid]] if weighted else torch.ones(int(valid.sum())))
    exp32[valid.nonzero()[:, 0], lab[valid]] = (-wl * inv) * gval
    dlc = dl.cpu()
    assert torch.isfinite(dlc).all()
    assert torch.equal(dlc, exp32)
    ref64 = torch.zeros(rows, ncls, dtype=torch.float64)
    ref64[valid.nonzero()[:, 0], lab[valid]] = -wv * gval / den
    r_d = ratio(dlc, ref64, 4.001 * U * ref64.abs() + 1e-300)
    print(f"nll {rows}x{ncls} w {weighted} g {gout}: loss {r_loss:.3f} wsum {r_ws:.3f} dlogp {r_d:.3f}")
    assert r_loss < 1 and r_ws < 1 and r_d < 1


# ----------------------------------------------------------------------------------------------------------------------
# Adam and the dropout multiply
# ----------------------------------------------------------------------------------------------------------------------
def _adam_grads(n, steps, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    mag = 10.0 ** (torch.rand(n, device="cuda", generator=g) * 11 - 8)          # 1e-8 ... 1e3
    sign = torch.where(torch.rand(n, device="cuda", generator=g) < 0.5, -1.0, 1.0)
    base = mag * sign
    for t in range(steps):
        gr = base * (0.5 + torch.rand(n, device="cuda", generator=g))
        gr[(torch.arange(n, device="cuda") + t) % 7 == 0] = 0.0              # exact zeros: denominator eps
        yield gr


@pytest.mark.parametrize("wd", [0.0, 1e-4], ids=["wd0", "wd1e-4"])
@pytest.mark.parametrize("n", [1, 1000, 606209])
def test_adam_step_matches_torch_adam(n, wd):
    """Each step from torch's state (p, m, v copied in), on the same gradient, against torch.optim.Adam's single-tensor
    CUDA step.  The betas are exact in fp32, so 1 - beta is the same number on both sides (the C ABI takes fp32 betas and
    forms 1 - beta in fp32; torch forms it from the Python double)."""
    L = _L()
    lr, b1, b2, eps = 1e-3, 0.875, 1 - 2.0 ** -10, 1e-8
    steps = 1000
    g0 = torch.Generator(device="cuda").manual_seed(n)
    p = torch.nn.Parameter(torch.randn(n, device="cuda", generator=g0))
    opt = torch.optim.Adam([p], lr=lr, betas=(b1, b2), eps=eps, weight_decay=wd, foreach=False, fused=False)
    kp, km, kv = torch.empty(n, device="cuda"), torch.empty(n, device="cuda"), torch.empty(n, device="cuda")
    worst_p = worst_mv = 0.0
    same_mv = 0
    for t, gr in enumerate(_adam_grads(n, steps, n + 1), start=1):
        st = opt.state.get(p)
        kp.copy_(p.detach())
        km.copy_(st["exp_avg"] if st else torch.zeros(n, device="cuda"))
        kv.copy_(st["exp_avg_sq"] if st else torch.zeros(n, device="cuda"))
        p.grad = gr.clone()
        opt.step()
        L.psg_adam_step(kp.data_ptr(), gr.data_ptr(), km.data_ptr(), kv.data_ptr(), n, lr, b1, b2, eps, wd, t, _st())
        st = opt.state[p]
        tm, tv = st["exp_avg"], st["exp_avg_sq"]
        dm = ((km - tm).abs().double() / _ulp_cuda(tm)).max().item()
        dv = ((kv - tv).abs().double() / _ulp_cuda(tv)).max().item()
        worst_mv = max(worst_mv, dm, dv)
        same_mv += int(torch.equal(km, tm) and torch.equal(kv, tv))
        # update magnitude from torch's new state: (lr / bc1) |m| / (sqrt(v / bc2) + eps)
        upd = (lr / (1 - b1 ** t)) * tm.double().abs() / (torch.sqrt(tv.double() / (1 - b2 ** t)) + eps)
        bound = 2 * _ulp_cuda(p.detach()) + 8 * U * upd
        worst_p = max(worst_p, ((kp - p.detach()).abs().double() / bound).max().item())
    print(f"adam n {n} wd {wd}: p {worst_p:.3f} of the gate; m, v {worst_mv:.1f} ulp at most, bit-identical on "
          f"{same_mv}/{steps} steps")
    assert worst_p < 1 and worst_mv <= 1


def _ulp_cuda(x):
    a = x.abs().float()
    return (torch.nextafter(a, torch.full_like(a, math.inf)) - a).double()


@pytest.mark.parametrize("n", [1000, 606209])
def test_adam_drift_against_fp64(n):
    """1000 free-running steps with the default betas against an fp64 restatement of the kernel's formula (the fp32
    hyper-parameters promoted): the parameters drift by no more than the roundings of each step allow."""
    L = _L()
    lr, b1, b2, eps, wd = 1e-3, 0.9, 0.999, 1e-8, 1e-4
    f = lambda v: float(np.float32(v))                            # noqa: E731
    lr_, b1_, b2_, eps_, wd_ = f(lr), f(b1), f(b2), f(eps), f(wd)
    steps = 1000
    p = torch.randn(n, device="cuda", generator=torch.Generator(device="cuda").manual_seed(3))
    m, v = torch.zeros_like(p), torch.zeros_like(p)
    pd, md, vd = p.double(), m.double(), v.double()
    budget = torch.zeros(n, dtype=torch.float64, device="cuda")
    for t, gr in enumerate(_adam_grads(n, steps, 7), start=1):
        L.psg_adam_step(p.data_ptr(), gr.data_ptr(), m.data_ptr(), v.data_ptr(), n, lr, b1, b2, eps, wd, t, _st())
        gd = gr.double() + wd_ * pd
        md = md + (gd - md) * (1 - b1_)
        vd = vd * b2_ + gd * gd * (1 - b2_)
        upd = (lr_ / (1 - b1_ ** t)) * md / (torch.sqrt(vd) / math.sqrt(1 - b2_ ** t) + eps_)
        pd = pd - upd
        # one rounding of p per step, and the update's relative error: v's recurrence keeps the roundings of the last
        # 1 / (1 - beta2) = 1000 steps, halved by the square root
        budget += 2 * U * pd.abs() + 1024 * U * upd.abs()
    r = ((p.double() - pd).abs() / (budget + 1e-300)).max().item()
    print(f"adam drift n {n}: {r:.3f} of the accumulated per-step bound")
    assert r < 1


@pytest.mark.parametrize("scale", [2.0, 1.7])
@pytest.mark.parametrize("case", [(1, 4), (129, 20), (1000, 128), (128 * 593 + 5, 64)], ids=lambda c: f"{c[0]}x{c[1]}")
def test_tl_mul_bitexact(case, scale):
    L = _L()
    rows, C = case
    g = _gen(rows + C)
    w = _wchunks(C)
    x = torch.randn(rows, C, generator=g)
    m = (torch.rand(rows, C, generator=g) < 0.5).float() * (1 + torch.rand(rows, C, generator=g))
    xt, mt = to_t(x, w), to_t(m, w)
    L.psg_tl_mul(xt.data_ptr(), w, mt.data_ptr(), w, rows, C, scale, _st())
    torch.cuda.synchronize()
    got = from_t(xt, rows, w)
    assert torch.equal(got[:rows, :C], x * (m * scale))
    assert torch.isnan(got[:, C:]).all(), "columns past C are not touched"


# ----------------------------------------------------------------------------------------------------------------------
# one layer composed as train.py composes it
# ----------------------------------------------------------------------------------------------------------------------
COMPOSE = [(12, 0, 32, True), (64, 256, 256, True), (128, 0, 13, False)]
COMPOSE_GATE = 1e-5


def _zero_t(x):
    return to_t(x, fill=0.0)


@pytest.mark.parametrize("rows", [1000, 65536])
@pytest.mark.parametrize("layer", COMPOSE, ids=["sa1_12to32", "fp_64+256to256", "conv2_128to13"])
def test_layer_composed_like_train(layer, rows):
    """psg_mlp_forward (mode 0) -> psg_bn_train_forward -> loss sum(y * R) -> psg_bn_train_backward (dz aliasing dy) ->
    psg_conv_wgrad -> psg_mlp_backward, in TrainEngine._conv_bn_relu / _chain_backward order, against fp64 autograd of
    linear + batch_norm(training=True) + relu, the ReLU mask taken from the kernel's y.  The GEMM operands are
    zero-padded as train.py allocates them."""
    L = _L()
    k1, k2, cout, has_bn = layer
    cin = k1 + k2
    g = _gen(rows + cin + cout)
    a1 = torch.randn(rows, k1, generator=g)
    a2 = torch.randn(rows, k2, generator=g) if k2 else None
    W = torch.randn(cout, cin, generator=g) / math.sqrt(cin)
    b = torch.randn(cout, generator=g) * 0.1
    gamma, beta = 0.5 + torch.rand(cout, generator=g), torch.randn(cout, generator=g) * 0.1
    R = torch.randn(rows, cout, generator=g)
    st = _st()
    h = L.psg_mlp_create_device(cin, cout)
    try:
        Wd, bd = W.cuda(), b.cuda()
        L.psg_mlp_load(h, Wd.data_ptr(), bd.data_ptr(), st)
        t1 = _zero_t(a1)
        t2 = _zero_t(a2) if k2 else None
        w1, w2, wo = _wchunks(k1), (_wchunks(k2) if k2 else 0), _wchunks(cout)
        zt = torch.zeros(((rows + 127) // 128) * 128 * 4 * wo, device="cuda")
        L.psg_mlp_forward(h, t1.data_ptr(), w1, 0, w1, t2.data_ptr() if k2 else None, w2, 0, w2, rows, zt.data_ptr(), wo, 0,
                          0, st)
        out = {}
        if has_bn:
            yt = torch.zeros_like(zt)
            mean, inv = torch.empty(cout, device="cuda"), torch.empty(cout, device="cuda")
            ws = torch.empty(L.psg_bn_workspace(cout), dtype=torch.uint8, device="cuda")
            gmd, btd = gamma.cuda(), beta.cuda()
            L.psg_bn_train_forward(zt.data_ptr(), wo, rows, cout, gmd.data_ptr(), btd.data_ptr(), None, None,
                                   0.1, 1e-5, yt.data_ptr(), wo, 1, mean.data_ptr(), inv.data_ptr(), ws.data_ptr(), ws.numel(), st)
            cur = _zero_t(R)                                         # dL/dy, then dz in place
            dg, dbt = torch.empty(cout, device="cuda"), torch.empty(cout, device="cuda")
            L.psg_bn_train_backward(cur.data_ptr(), wo, yt.data_ptr(), wo, zt.data_ptr(), wo, rows, cout, gmd.data_ptr(),
                                    mean.data_ptr(), inv.data_ptr(), dg.data_ptr(), dbt.data_ptr(), cur.data_ptr(), wo,
                                    ws.data_ptr(), ws.numel(), st)
            out["y"] = from_t(yt, rows, wo)[:rows, :cout]
            out["dgamma"], out["dbeta"] = dg, dbt
        else:
            cur = _zero_t(R)
            out["z"] = from_t(zt, rows, wo)[:rows, :cout]
        dW, db = torch.empty(cout, cin, device="cuda"), torch.empty(cout, device="cuda")
        ws2 = torch.empty(L.psg_wgrad_workspace(cout, cin, rows), dtype=torch.uint8, device="cuda")
        L.psg_conv_wgrad(cur.data_ptr(), wo, cout, t1.data_ptr(), w1, 0, k1 if not k2 else 4 * w1, t2.data_ptr() if k2 else None,
                         w2, 0, 4 * w2 if k2 else 0, rows, dW.data_ptr(), db.data_ptr(), 0, ws2.data_ptr(), ws2.numel(), st)
        kin = 4 * (w1 + w2)
        dxt = torch.zeros(((rows + 127) // 128) * 128 * kin, device="cuda")
        L.psg_mlp_backward(h, cur.data_ptr(), wo, rows, dxt.data_ptr(), kin // 4, None, 0, 0, st)
        torch.cuda.synchronize()
    finally:
        L.psg_mlp_destroy(h)
    dx = from_t(dxt, rows, kin // 4)[:rows]
    dx = torch.cat([dx[:, :k1], dx[:, 4 * w1: 4 * w1 + k2]], 1) if k2 else dx[:, :k1]
    # fp64 reference
    x = (torch.cat([a1, a2], 1) if k2 else a1).double().requires_grad_(True)
    Wr, br = W.double().requires_grad_(True), b.double().requires_grad_(True)
    gr, be = gamma.double().requires_grad_(True), beta.double().requires_grad_(True)
    z = x @ Wr.t() + br
    errs = {}
    if has_bn:
        yb = torch.nn.functional.batch_norm(z, None, None, gr, be, training=True, eps=float(np.float32(1e-5)))
        y = yb * (out["y"].double() > 0)                              # the kernel's ReLU routing
        (y * R.double()).sum().backward()
        errs["y"] = _relf(out["y"], y.detach())
        errs["dgamma"] = _relf(out["dgamma"].cpu(), gr.grad)
        errs["dbeta"] = _relf(out["dbeta"].cpu(), be.grad)
    else:
        (z * R.double()).sum().backward()
        errs["z"] = _relf(out["z"], z.detach())
        errs["db"] = _relf(db.cpu(), br.grad)
    errs["dW"] = _relf(dW.cpu(), Wr.grad)
    errs["dx"] = _relf(dx, x.grad)
    print(f"layer {layer} rows {rows}: " + " ".join(f"{k} {v:.2e}" for k, v in errs.items()))
    assert max(errs.values()) < COMPOSE_GATE, errs


def _relf(got, ref):
    got = got.double().cpu()
    assert torch.isfinite(got).all()
    return ((got - ref).norm() / ref.norm()).item()


# ----------------------------------------------------------------------------------------------------------------------
# determinism
# ----------------------------------------------------------------------------------------------------------------------
def test_every_op_is_deterministic():
    """DESIGN.md section 10: each op called twice on the same inputs gives bit-identical outputs."""
    L = _L()
    rows, C, st = 128 * 593 + 5, 64, _st()
    g = _gen(99)
    z, dy = torch.randn(rows, C, generator=g), torch.randn(rows, C, generator=g)
    y = torch.relu(torch.randn(rows, C, generator=g))
    a = torch.randn(rows, 20, generator=g)
    w = _wchunks(C)
    zt, yt0, a1t = to_t(z, w), to_t(y, w), to_t(a, 8)
    gam, bet = torch.rand(C, device="cuda") + 0.5, torch.randn(C, device="cuda")
    ws = torch.empty(max(L.psg_bn_workspace(C), L.psg_wgrad_workspace(C, 20, rows), L.psg_nll_workspace()),
                     dtype=torch.uint8, device="cuda")

    def run():
        o = {}
        yt, sm, si = torch.zeros_like(zt), torch.empty(C, device="cuda"), torch.empty(C, device="cuda")
        rm, rv = torch.zeros(C, device="cuda"), torch.ones(C, device="cuda")
        L.psg_bn_train_forward(zt.data_ptr(), w, rows, C, gam.data_ptr(), bet.data_ptr(), rm.data_ptr(), rv.data_ptr(), 0.1,
                               1e-5, yt.data_ptr(), w, 1, sm.data_ptr(), si.data_ptr(), ws.data_ptr(), ws.numel(), st)
        o.update(y=yt, sm=sm, si=si, rm=rm, rv=rv)
        dzt, dg, db = to_t(dy, w), torch.empty(C, device="cuda"), torch.empty(C, device="cuda")
        L.psg_bn_train_backward(dzt.data_ptr(), w, yt0.data_ptr(), w, zt.data_ptr(), w, rows, C, gam.data_ptr(), sm.data_ptr(),
                                si.data_ptr(), dg.data_ptr(), db.data_ptr(), dzt.data_ptr(), w, ws.data_ptr(), ws.numel(), st)
        o.update(dz=dzt, dg=dg, db=db)
        dW, dbias = torch.empty(C, 20, device="cuda"), torch.empty(C, device="cuda")
        L.psg_conv_wgrad(dzt.data_ptr(), w, C, a1t.data_ptr(), 8, 0, 20, None, 0, 0, 0, rows, dW.data_ptr(), dbias.data_ptr(), 0,
                         ws.data_ptr(), ws.numel(), st)
        o.update(dW=dW, dbias=dbias)
        logp = torch.empty(rows, 13, device="cuda")
        L.psg_log_softmax_rows(zt.data_ptr(), w, rows, 13, logp.data_ptr(), st)
        dlz = torch.zeros(rows // 128 * 128 + 128, 16, device="cuda")
        L.psg_dlogits_from_dlogp(zt.data_ptr(), w, logp.data_ptr(), rows, 13, dlz.data_ptr(), 4, st)
        lab = (torch.arange(rows, device="cuda") * 7) % 15 - 1
        nl = torch.empty(2, device="cuda")
        L.psg_nll_loss(logp.data_ptr(), lab.data_ptr(), None, rows, 13, nl.data_ptr(), nl[1:].data_ptr(), ws.data_ptr(),
                       ws.numel(), st)
        dl = torch.empty(rows, 13, device="cuda")
        L.psg_nll_loss_backward(lab.data_ptr(), None, rows, 13, None, nl[1:].data_ptr(), dl.data_ptr(), st)
        o.update(logp=logp, dlz=dlz, nl=nl, dl=dl)
        p, m, v = dW.flatten().clone(), torch.zeros(C * 20, device="cuda"), torch.zeros(C * 20, device="cuda")
        for t in (1, 2):
            L.psg_adam_step(p.data_ptr(), dW.data_ptr(), m.data_ptr(), v.data_ptr(), C * 20, 1e-3, 0.9, 0.999, 1e-8, 1e-4, t, st)
        o.update(p=p, m=m, v=v)
        torch.cuda.synchronize()
        return o

    a_, b_ = run(), run()
    for k in a_:
        assert torch.equal(a_[k].view(torch.int32), b_[k].view(torch.int32)), k


# ----------------------------------------------------------------------------------------------------------------------
# view widths: rejected before anything is launched
# ----------------------------------------------------------------------------------------------------------------------
def test_narrow_views_are_rejected():
    """Each call names a view narrower than the columns it would be read or written for.  The buffers are allocated for
    the widest interpretation, so even a missing check would stay inside them."""
    L = _L()
    st, rows = _st(), 1000
    rpad = 1024
    big = lambda cols: torch.zeros(rpad * cols + 4096, device="cuda")   # noqa: E731
    A, B, D, Y = big(64), big(64), big(64), big(64)
    vec = torch.zeros(1024, device="cuda")
    ws = torch.zeros(max(L.psg_bn_workspace(64), L.psg_wgrad_workspace(64, 64, rows)), dtype=torch.uint8, device="cuda")
    dW = torch.zeros(64 * 64, device="cuda")

    def wgrad(dzw, cout, a1w, a1c0, k1, a2w=0, a2c0=0, k2=0, db=True):
        L.psg_conv_wgrad(D.data_ptr(), dzw, cout, A.data_ptr(), a1w, a1c0, k1, B.data_ptr() if k2 else None, a2w, a2c0, k2, rows,
                         dW.data_ptr(), vec.data_ptr() if db else None, 0, ws.data_ptr(), ws.numel(), st)

    wgrad(4, 13, 4, 0, 13)                                             # a valid call first
    bad = [
        lambda: wgrad(2, 13, 4, 0, 13),                                # dz narrower than cout, with db
        lambda: wgrad(2, 13, 4, 0, 13, db=False),                      # and without
        lambda: wgrad(4, 13, 4, 2, 12),                                # a1_c0 + ceil(k1 / 4) > a1_wchunks
        lambda: wgrad(4, 13, 4, 0, 20),
        lambda: wgrad(4, 13, 4, 0, 16, 4, 1, 13),                      # the same for A2
        lambda: wgrad(4, 13, 8, 0, 16, 4, 0, 20),
        lambda: L.psg_bn_train_forward(A.data_ptr(), 4, rows, 32, vec.data_ptr(), vec.data_ptr(), None, None, 0.1, 1e-5,
                                       Y.data_ptr(), 8, 1, vec.data_ptr(), vec.data_ptr(), ws.data_ptr(), ws.numel(), st),
        lambda: L.psg_bn_train_forward(A.data_ptr(), 8, rows, 32, vec.data_ptr(), vec.data_ptr(), None, None, 0.1, 1e-5,
                                       Y.data_ptr(), 4, 1, vec.data_ptr(), vec.data_ptr(), ws.data_ptr(), ws.numel(), st),
    ]
    for narrow in ("dy", "y", "z", "dz"):
        wv = {k: (4 if k == narrow else 8) for k in ("dy", "y", "z", "dz")}
        bad.append(lambda wv=wv: L.psg_bn_train_backward(A.data_ptr(), wv["dy"], Y.data_ptr(), wv["y"], B.data_ptr(), wv["z"], rows,
                                                         32, vec.data_ptr(), vec.data_ptr(), vec.data_ptr(), vec.data_ptr(),
                                                         vec.data_ptr(), D.data_ptr(), wv["dz"], ws.data_ptr(), ws.numel(), st))
    bad += [
        lambda: L.psg_tl_mul(A.data_ptr(), 4, B.data_ptr(), 8, rows, 32, 2.0, st),
        lambda: L.psg_tl_mul(A.data_ptr(), 8, B.data_ptr(), 4, rows, 32, 2.0, st),
        lambda: L.psg_log_softmax_rows(A.data_ptr(), 3, rows, 13, D.data_ptr(), st),
        lambda: L.psg_dlogits_from_dlogp(A.data_ptr(), 3, B.data_ptr(), rows, 13, D.data_ptr(), 4, st),
        lambda: L.psg_dlogits_from_dlogp(A.data_ptr(), 4, B.data_ptr(), rows, 5, D.data_ptr(), 2, st),
    ]
    before = L.psg_launch_count()
    for call in bad:
        with pytest.raises(L.PsgError, match="invalid argument"):
            call()
    assert L.psg_launch_count() == before, "a rejected call launched work"
    torch.cuda.synchronize()


# ----------------------------------------------------------------------------------------------------------------------
# BatchNorm momentum=None through the training engine
# ----------------------------------------------------------------------------------------------------------------------
def test_bn_momentum_none_is_cumulative_average():
    """nn.BatchNorm with momentum=None keeps the cumulative average of the batch statistics (factor
    1 / num_batches_tracked, counted after the increment)."""
    from pointsecguard_b200 import synthetic as syn
    from pointsecguard_b200.models.pointnet2_sem_seg import get_model
    from pointsecguard_b200.train import TrainEngine
    m = get_model(13)
    m.load_state_dict(syn.make_state_dict("ssg", init="he"))
    m = m.cuda().train()
    for mod in m.modules():
        if isinstance(mod, torch.nn.modules.batchnorm._BatchNorm):
            mod.momentum = None
    eng = TrainEngine(m)
    bn = m.bn1
    seen = []
    torch.manual_seed(0)
    for s in range(2):
        x, _ = syn.make_painted_blocks(1, 1024, 70 + s)
        eng.forward(x.cuda())
        r1 = eng.ctx["r1"]
        z = from_t(r1["z"].buf, 1024, r1["z"].wchunks)[:1024, :bn.num_features].double()
        seen.append((r1["mean"].cpu().double(), z.var(0, unbiased=True)))
        torch.cuda.synchronize()
        rm, rv = bn.running_mean.cpu().double(), bn.running_var.cpu().double()
        mean_ref = sum(a for a, _ in seen) / len(seen)
        mean_mag = sum(a.abs() for a, _ in seen) / len(seen)          # the saved means are fp32, the kernel's double
        var_ref = sum(v for _, v in seen) / len(seen)
        assert int(bn.num_batches_tracked) == s + 1
        assert ((rm - mean_ref).abs() <= 2 * ulp(mean_mag) + 1e-300).all(), s
        assert ((rv - var_ref).abs() <= 8 * ulp(var_ref)).all(), s
        if s == 0:
            assert torch.equal(bn.running_mean.cpu(), r1["mean"].cpu())
