"""Direct numerics tests of the sm_100a kernels against plain PyTorch fp32 references."""
import numpy
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ext():
    from veles.znicz_b200.kernels import load_extension
    return load_extension(required=True)


def _rel(a, b):
    a = a.float()
    b = b.float()
    return float((a - b).abs().max() / (b.abs().max() + 1e-12))


@pytest.mark.parametrize("engine", [0, 1])
@pytest.mark.parametrize("M,N,K", [(100, 10, 1024), (128, 128, 64), (300, 72, 200),
                                   (1999, 5625, 1776), (64, 791, 1392), (257, 32, 800)])
def test_gemm_nt_bias_act(ext, engine, M, N, K):
    """out = relu(a @ b^T + bias): FC forward shape family (/root/reference/
    tests/unit/test_all2all.py:98 perf shape 1999x1777->5625 rounded to K%8==0)."""
    torch.manual_seed(0)
    dev = "cuda"
    a = torch.randn(M, K, device=dev).bfloat16()
    b = (torch.randn(N, K, device=dev) / K ** 0.5).bfloat16()
    bias = torch.randn(N, device=dev)
    ref = torch.relu(a.float() @ b.float().t() + bias)
    for out_dt in (torch.bfloat16, torch.float32):
        # out-of-bounds guard of the reference's unit tests (tests/unit/test_gd.py:137-141): the
        # buffer is twice as large and NaN-filled; whatever lies behind the result must stay NaN
        big = torch.full((2 * M, N), float("nan"), device=dev, dtype=out_dt)
        out = big[:M]
        r = ext.gemm(a, K, False, b, K, True, out, N, False, M, N, K, bias, 3, 1.0, 0.0, 1, 0,
                     engine)
        assert r == 0
        torch.cuda.synchronize()
        assert _rel(out, ref) < (2e-2 if out_dt == torch.bfloat16 else 2e-3), (engine, out_dt)
        assert torch.isnan(big[M:]).all(), (engine, out_dt)


@pytest.mark.parametrize("engine", [0, 1])
@pytest.mark.parametrize("M,N,K", [(100, 1024, 16), (256, 64, 64), (130, 200, 72),
                                   (100, 1392, 792)])
def test_gemm_nn_alpha_beta(ext, engine, M, N, K):
    """err_in = alpha * err @ W + beta * err_in  (B stored [K][N], MN-major operand)."""
    torch.manual_seed(1)
    dev = "cuda"
    a = torch.randn(M, K, device=dev).bfloat16()
    b = (torch.randn(K, N, device=dev) / K ** 0.5).bfloat16()
    old = torch.randn(M, N, device=dev)
    ref = 0.5 * (a.float() @ b.float()) + 2.0 * old
    out = old.clone()
    r = ext.gemm(a, K, False, b, N, False, out, N, False, M, N, K, None, 0, 0.5, 2.0, 1, 0, engine)
    assert r == 0
    torch.cuda.synchronize()
    assert _rel(out, ref) < 3e-3


@pytest.mark.parametrize("engine", [0, 1])
@pytest.mark.parametrize("M,N,K,splits", [(64, 1024, 100, 1), (792, 1392, 104, 1),
                                           (32, 800, 25600, 8), (128, 128, 1000, 3)])
def test_gemm_tn_splitk(ext, engine, M, N, K, splits):
    """gradW = err^T @ x with both operands MN-major and fp32 split-K partials."""
    torch.manual_seed(2)
    dev = "cuda"
    a = torch.randn(K, M, device=dev).bfloat16()      # stored [K][M]
    b = torch.randn(K, N, device=dev).bfloat16()      # stored [K][N]
    ref = a.float().t() @ b.float()
    parts = torch.full((splits, M, N), float("nan"), device=dev)
    r = ext.gemm(a, M, True, b, N, False, parts, N, False, M, N, K, None, 0, 1.0, 0.0, splits,
                 M * N, engine)
    assert r == 0
    torch.cuda.synchronize()
    assert _rel(parts.sum(0), ref) < 2e-3


def _conv_ref(x, w, bias, ky, kx, pad, stride):
    # x NHWC, w [F][ky*kx*C]; pad = (L, T, R, B), stride = (sx, sy)
    n, h, ww, c = x.shape
    f = w.shape[0]
    xp = torch.nn.functional.pad(x.permute(0, 3, 1, 2), (pad[0], pad[2], pad[1], pad[3]))
    wt = w.view(f, ky, kx, c).permute(0, 3, 1, 2)
    y = torch.nn.functional.conv2d(xp, wt, bias, stride=(stride[1], stride[0]))
    return y.permute(0, 2, 3, 1).contiguous()


CONV_CASES = [
    # N, H, W, C, F, ky, kx, pad(L,T,R,B), stride(x,y)
    (4, 32, 32, 3, 32, 5, 5, (2, 2, 2, 2), (1, 1)),     # CIFAR conv1
    (4, 16, 16, 32, 32, 5, 5, (2, 2, 2, 2), (1, 1)),    # CIFAR conv2
    (3, 8, 8, 32, 64, 5, 5, (2, 2, 2, 2), (1, 1)),      # CIFAR conv3
    (2, 12, 12, 64, 88, 5, 5, (0, 0, 0, 0), (1, 1)),    # MNIST conv2-like
    (2, 15, 13, 8, 16, 3, 2, (1, 0, 2, 1), (2, 1)),     # odd geometry
    (2, 27, 27, 16, 24, 11, 11, (0, 0, 0, 0), (4, 4)),  # AlexNet conv1-like stride 4
    (2, 9, 9, 128, 128, 3, 3, (1, 1, 1, 1), (1, 1)),    # 64-channel slices of one tap (tpk = 1)
    (3, 20, 20, 8, 32, 5, 5, (2, 2, 2, 2), (1, 1)),     # channel-padded first layer (tpk = 8)
    (40, 32, 32, 8, 32, 5, 5, (2, 2, 2, 2), (1, 1)),   # CIFAR conv1 fprop: 320 CTAs x 4 k-blocks, 3-stage ring
    (2, 10, 10, 16, 16, 3, 3, (1, 1, 1, 1), (1, 1)),    # tpk = 4, dgrad with F = 16
    # TMA im2col operand (C % 64 == 0 fprop / wgrad, F % 64 == 0 stride-1 dgrad)
    (3, 14, 17, 64, 64, 3, 5, (2, 1, 1, 0), (1, 1)),    # asymmetric padding, tiles span images
    (2, 16, 16, 64, 64, 3, 3, (1, 1, 1, 1), (2, 2)),    # strided windows (dgrad stays on gather)
    (5, 13, 13, 192, 128, 3, 3, (1, 1, 1, 1), (1, 1)),  # AlexNet conv3-like, 3 channel slices / tap
    # large layers: 2-CTA persistent kernel (gemm_pair.cu) with the TMA im2col operand
    (8, 13, 13, 128, 256, 3, 3, (1, 1, 1, 1), (1, 1)),  # fprop BN 256; dgrad N = 128
    (4, 20, 20, 64, 384, 5, 5, (2, 2, 2, 2), (1, 1)),   # fprop 3 N-tiles of 128
    (3, 20, 21, 256, 128, 3, 3, (1, 1, 1, 1), (1, 1)),  # dgrad BN 256, ragged M
    (5, 31, 31, 64, 128, 5, 5, (2, 2, 2, 2), (2, 2)),   # strided fprop on the pair kernel
    (16, 20, 20, 64, 128, 3, 3, (1, 1, 1, 1), (1, 1)),  # pair wgrad: F = 128 (idle peer CTA), ragged Kw
    (12, 19, 19, 128, 256, 3, 3, (1, 1, 1, 1), (1, 1)), # pair wgrad with split-K, F = 256
]


@pytest.mark.parametrize("engine", [0, 1])
@pytest.mark.parametrize("case", CONV_CASES)
def test_conv_fprop_dgrad_wgrad(ext, engine, case):
    n, h, w_, c, f, ky, kx, pad, stride = case
    torch.manual_seed(3)
    dev = "cuda"
    tma0, pair0 = ext.im2col_tma_launches(), ext.conv_pair_launches()
    oh = 1 + (h - ky + pad[1] + pad[3]) // stride[1]
    ow = 1 + (w_ - kx + pad[0] + pad[2]) // stride[0]
    kw = ky * kx * c
    x = torch.randn(n, h, w_, c, device=dev).bfloat16()
    wm = (torch.randn(f, kw, device=dev) / kw ** 0.5)
    wq = wm.bfloat16().float()
    bias = torch.randn(f, device=dev)
    g = [n, h, w_, c, oh, ow, f, ky, kx, stride[1], stride[0], pad[1], pad[0]]
    xr = x.float().requires_grad_(True)
    wr = wq.clone().requires_grad_(True)
    ref = _conv_ref(xr, wr, bias, ky, kx, pad, stride)
    eo = torch.randn_like(ref).bfloat16()
    ref.backward(eo.float())
    # fprop
    big_out = torch.full((2 * n, oh, ow, f), float("nan"), device=dev, dtype=torch.bfloat16)
    out = big_out[:n]                      # out-of-bounds guard: the second half must stay NaN
    if engine == 1:
        ld = (kw + 7) // 8 * 8
        wlp = torch.zeros(f, ld, device=dev, dtype=torch.bfloat16)
        wlp[:, :kw] = wq.bfloat16()
        r = ext.conv_fprop(x, wlp, ld, False, bias, out, g, 0, 1)
    else:
        r = ext.conv_fprop(x, wq.contiguous(), kw, False, bias, out, g, 0, 0)
    assert r == 0
    torch.cuda.synchronize()
    assert _rel(out, ref.detach()) < 2e-2
    assert torch.isnan(big_out[n:]).all()
    # dgrad
    ei = torch.full((n, h, w_, c), float("nan"), device=dev, dtype=torch.bfloat16)
    if engine == 1:
        cp = (c + 7) // 8 * 8
        wd = torch.zeros(ky * kx * f, cp, device=dev, dtype=torch.bfloat16)
        wd.view(ky * kx, f, cp)[:, :, :c] = wq.view(f, ky * kx, c).permute(1, 0, 2).bfloat16()
        r = ext.conv_dgrad(eo, wd, cp, False, ei, g, 1.0, 0.0, 1, None, 0)
        if r == 0 and c % 8 == 0:
            # the same dgrad with the producer's strict-ReLU derivative folded into the epilogue
            ei2 = torch.empty_like(ei)
            xin = torch.randn(n, h, w_, c, device=dev).bfloat16()
            r2 = ext.conv_dgrad(eo, wd, cp, False, ei2, g, 1.0, 0.0, 1, xin, 3)
            assert r2 == 0
            torch.cuda.synchronize()
            assert torch.equal(ei2, (ei.float() * (xin.float() > 0)).bfloat16())
    else:
        r = ext.conv_dgrad(eo, wq.contiguous(), kw, False, ei, g, 1.0, 0.0, 0, None, 0)
    assert r == 0
    torch.cuda.synchronize()
    assert _rel(ei, xr.grad) < 2e-2
    # wgrad
    if engine == 1 and f % 8:
        return
    splits = int(ext.pick_splits(kw, f, n * oh * ow, 16)) if engine == 1 else 4
    parts = torch.full((splits, f, kw), float("nan"), device=dev)
    bparts = torch.full((splits, f), float("nan"), device=dev) if engine == 1 else None
    r = ext.conv_wgrad(eo, x, parts, splits, g, False, engine, bparts)
    assert r in (0, 1)
    torch.cuda.synchronize()
    assert torch.isfinite(parts).all()           # every split-K partial slot was written
    assert _rel(parts.sum(0), wr.grad) < 5e-3
    if r == 1:      # bias gradient delivered as the extra "ones" row of the product
        ref_b = eo.float().reshape(-1, f).sum(0)
        assert _rel(bparts.sum(0), ref_b) < 5e-3
    if engine == 1:
        # the TMA im2col producer really ran where the geometry allows it (no silent fallback)
        f_pair = c % 64 == 0 and f >= 128 and n * oh * ow >= 1024
        d_pair = f % 64 == 0 and stride == (1, 1) and c >= 128 and n * h * w_ >= 1024
        d_tma = f % 64 == 0 and stride == (1, 1) and not d_pair
        w_pair = c % 64 == 0 and f % 128 == 0 and n * oh * ow >= 4096
        want_pair = int(f_pair) + 2 * int(d_pair) + int(w_pair)   # (dgrad runs twice: plain + folded f')
        want_tma = (1 if (c % 64 == 0 and not f_pair) else 0) + \
            (2 if (d_tma and c % 8 == 0) else int(d_tma))
        got = (ext.conv_pair_launches() - pair0, ext.im2col_tma_launches() - tma0)
        assert got == (want_pair, want_tma), (got, want_pair, want_tma)


def test_fused_update_matches_reference_formula(ext):
    """K3/K4 semantics (/root/reference/cuda/gradient_descent.store_output.cu)."""
    torch.manual_seed(4)
    dev = "cuda"
    rows, cols = 37, 53
    w = torch.randn(rows, cols, device=dev)
    g = torch.randn(3, rows, cols, device=dev)
    acc = torch.randn(rows, cols, device=dev)
    vel = torch.randn(rows, cols, device=dev)
    hyper = torch.tensor([0.1, 0.01, 0.3, 0.9, 0.5, 0.25, 0.75, 0.8, 0.002, 0, 0, 0, 0, 0, 0, 0],
                         device=dev)
    cs = w.sum(0)
    w0, acc0, vel0 = w.clone(), acc.clone(), vel.clone()
    lp = torch.zeros(rows, 56, device=dev, dtype=torch.bfloat16)
    gout = torch.zeros(rows, cols, device=dev)
    ext.fused_update(w, [g.data_ptr()], 3, rows * cols, gout, acc, vel, hyper, cs,
                     1 | 2 | 4 | 8, False, rows, cols, lp, 56, None, 0, 0, 0, [], 0, 0, 0, 0, 0)
    torch.cuda.synchronize()
    gs = g.sum(0)
    lr, wd, l1, mom, aa, ab, ga, gb, ortho = [float(v) for v in hyper[:9]]
    gd = -lr * (gs + wd * ((1 - l1) * w0 + 0.5 * l1 * torch.sign(w0)) +
                ortho / rows * (cs - w0))
    a = ab * acc0 + aa * gd
    gd = gd * gb + ga * a
    gd = gd + vel0 * mom
    assert _rel(gout, gs) < 1e-6
    assert _rel(acc, a) < 1e-5
    assert _rel(vel, gd) < 1e-5
    assert _rel(w, w0 + gd) < 1e-5
    assert _rel(lp[:, :cols], (w0 + gd)) < 1e-2


def test_multi_update_matches_per_tensor_update(ext):
    """The whole-network step kernel must be bit-compatible (fixed summation order aside)
    with the per-tensor fused update: weights with ortho + split-K partials, a conv tensor
    with channel-padded gradients and both bf16 shadows, and a bias with 128 partials that
    takes the lane-cooperative path."""
    torch.manual_seed(11)
    dev = "cuda"
    hyper = torch.tensor([0.1, 0.01, 0.3, 0.9, 0.5, 0.25, 0.75, 0.8, 0.002,
                          0.2, 0.0, 0.0, 0.7, 0, 0, 0], device=dev)

    def P(t):
        return 0 if t is None else t.data_ptr()
    specs = []
    # (rows, cols, nparts, flags, is_bias, conv(taps, C, c_pad, lp_cpad, g_cpad), lanes)
    specs.append(dict(rows=37, cols=53, nparts=3, flags=1 | 2 | 4 | 8, bias=False, conv=None,
                      lanes=2))
    specs.append(dict(rows=32, cols=75, nparts=22, flags=1 | 2 | 8, bias=False,
                      conv=(25, 3, 8, 8, 8), lanes=16))
    specs.append(dict(rows=1, cols=32, nparts=128, flags=1 | 2, bias=True, conv=None, lanes=32))
    specs.append(dict(rows=64, cols=800, nparts=5, flags=1 | 2 | 8, bias=False,
                      conv=(25, 32, 32, 0, 0), lanes=1))
    # >= 2^20 elements: the 4-elements-per-thread tile path (FC6-sized tensors)
    specs.append(dict(rows=1030, cols=1048, nparts=2, flags=1 | 2 | 4, bias=False, conv=None,
                      lanes=1))
    # float4 path with per-element shadows (conv-shaped 1.33 M weights, bf16 [tap][F][C] shadow)
    specs.append(dict(rows=384, cols=3456, nparts=3, flags=1 | 2 | 8, bias=False,
                      conv=(9, 384, 384, 0, 0), lanes=1))
    # float4 chunks that straddle rows (cols % 4 != 0)
    specs.append(dict(rows=1031, cols=1049, nparts=1, flags=1 | 2, bias=False, conv=None,
                      lanes=1))
    ref, new, descs = [], [], []
    for sp in specs:
        rows, cols = sp["rows"], sp["cols"]
        conv = sp["conv"]
        g_cpad = conv[4] if conv else 0
        gcols = conv[0] * g_cpad if g_cpad else cols
        w = torch.randn(rows, cols, device=dev)
        g = torch.randn(sp["nparts"], rows, gcols, device=dev)
        acc = torch.randn(rows, cols, device=dev) if sp["flags"] & 4 else None
        vel = torch.randn(rows, cols, device=dev)
        ld = ((cols + 7) // 8) * 8
        taps = C = c_pad = lp_cpad = 0
        lp_conv = None
        if conv:
            taps, C, c_pad, lp_cpad, _ = conv
            if lp_cpad:
                ld = taps * lp_cpad
        lp = None if sp["bias"] else torch.zeros(rows, ld, device=dev, dtype=torch.bfloat16)
        if conv:
            lp_conv = torch.zeros(taps * rows, c_pad, device=dev, dtype=torch.bfloat16)
        two = []
        for _ in range(2):
            two.append(dict(w=w.clone(), acc=None if acc is None else acc.clone(),
                            vel=vel.clone(), gout=torch.zeros(rows, cols, device=dev),
                            cs=torch.zeros(cols, device=dev),
                            lp=None if lp is None else lp.clone(),
                            lp_conv=None if lp_conv is None else lp_conv.clone()))
        a, b = two
        if sp["flags"] & 8:
            ext.col_sums(a["w"], a["cs"], rows, cols, False)
        ext.fused_update(a["w"], [g.data_ptr()], sp["nparts"], rows * gcols, a["gout"], a["acc"],
                         a["vel"], hyper, a["cs"] if sp["flags"] & 8 else None, sp["flags"],
                         sp["bias"], rows, cols, a["lp"], ld, a["lp_conv"], taps, C, c_pad,
                         [], 0, 0, 0, lp_cpad, g_cpad)
        descs.append([P(b["w"]), P(b["gout"]), P(b["acc"]), P(b["vel"]), P(hyper),
                      P(b["cs"]) if sp["flags"] & 8 else 0, g.data_ptr(), 0, 0, 0, 0, 0, 0, 0,
                      rows * gcols, rows * cols, sp["nparts"], g_cpad, sp["flags"],
                      1 if sp["bias"] else 0, rows, cols, sp["lanes"], 1,
                      P(b["lp"]), ld, lp_cpad, P(b["lp_conv"]), taps, C, c_pad])
        ref.append(a)
        new.append(b)
        sp["g"] = g
    packed, tiles, red = ext.multi_update_table(descs, 0)
    assert red == sum((d[15] + 3) // 4 * 4 for d in descs)     # 16-byte aligned slots
    table = packed.cuda()
    sync = torch.zeros(2, dtype=torch.int32, device=dev)
    for _ in range(1):
        ext.multi_update(table, len(descs), tiles, True, [], 0, 0, sync, [], 0, 1, [], 0, 0, 0, 0)
    torch.cuda.synchronize()
    assert int(sync[0]) == 0 and int(sync[1]) == 1      # one grid barrier generation
    for a, b, sp in zip(ref, new, specs):
        for k in ("w", "vel", "gout", "acc"):
            if a[k] is None:
                continue
            assert _rel(b[k], a[k]) < 2e-6, (sp["rows"], sp["cols"], k)
        for k in ("lp", "lp_conv"):
            if a[k] is not None:
                assert _rel(b[k].float(), a[k].float()) < 1e-2, (sp["rows"], k)
                assert float(b[k].float().abs().sum()) > 0
    # disabled tensors must be left alone; a second launch must work (barrier re-arms)
    descs[0][23] = 0
    packed, tiles2, _ = ext.multi_update_table(descs, 0)
    assert tiles2 == tiles
    table.copy_(packed)
    w_before = new[0]["w"].clone()
    ext.multi_update(table, len(descs), tiles, True, [], 0, 0, sync, [], 0, 1, [], 0, 0, 0, 0)
    torch.cuda.synchronize()
    assert torch.equal(new[0]["w"], w_before)
    assert int(sync[1]) == 2


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("n_out,act,softmax", [(10, 0, True), (7, 1, False), (16, 3, False),
                                               (3, 4, False)])
def test_fc_small_forward(ext, dtype, n_out, act, softmax):
    torch.manual_seed(n_out)
    dev = "cuda"
    batch, n_in = 37, 1000
    x = torch.randn(batch, n_in, device=dev).to(dtype)
    w = torch.randn(n_out, n_in, device=dev) * 0.05
    b = torch.randn(n_out, device=dev)
    out = torch.full((batch, n_out), float("nan"), device=dev,
                     dtype=torch.float32 if softmax else dtype)
    mi = torch.full((batch,), -1, device=dev, dtype=torch.int32)
    ext.fc_small_forward(x, w, b, out, mi if softmax else None, batch, n_in, n_out, act, softmax,
                         [])
    torch.cuda.synchronize()
    z = x.float() @ w.t() + b
    if softmax:
        ref = torch.softmax(z, dim=1)
        assert torch.equal(mi.long(), z.argmax(dim=1))
    else:
        ref = {1: lambda t: 1.7159 * torch.tanh(0.6666 * t), 3: torch.relu,
               4: torch.sigmoid}[act](z)
    assert _rel(out.float(), ref) < (1e-5 if dtype == torch.float32 and softmax else 2e-2 if dtype == torch.bfloat16 else 1e-5)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("n_out,act", [(10, 0), (7, 1), (16, 3)])
def test_fc_small_backward(ext, dtype, n_out, act):
    torch.manual_seed(100 + n_out)
    dev = "cuda"
    batch, n_in, bsplit = 53, 520, 4
    x = torch.randn(batch, n_in, device=dev).to(dtype)
    w = torch.randn(n_out, n_in, device=dev) * 0.05
    y = torch.randn(batch, n_out, device=dev).to(dtype)
    err = torch.randn(batch, n_out, device=dev).to(dtype)
    ei = torch.randn(batch, n_in, device=dev).to(dtype)
    ei0, err0 = ei.clone(), err.clone()
    gw = torch.full((bsplit, n_out, n_in), float("nan"), device=dev)
    gb = torch.full((bsplit, n_out), float("nan"), device=dev)
    alpha, beta = 0.75, 0.5
    ext.fc_small_backward(err, y if act else None, x, w, ei, gw, gb, batch, n_in, n_out, act,
                          alpha, beta, bsplit)
    torch.cuda.synchronize()
    yf = y.float()
    d = {0: torch.ones_like(yf), 1: yf * yf * (-0.388484177) + 1.14381894,
         3: (yf > 0).float()}[act]
    e = err0.float() * d
    tol = 1e-5 if dtype == torch.float32 else 2e-2
    assert torch.equal(err, err0)               # err_output is read-only for the kernel
    assert _rel(ei.float(), alpha * (e @ w) + beta * ei0.float()) < tol
    assert _rel(gw.sum(0), e.t() @ x.float()) < tol
    assert _rel(gb.sum(0), e.sum(0)) < tol
    # optional outputs
    ext.fc_small_backward(err0.clone(), y if act else None, x, w, None, None, None, batch, n_in,
                          n_out, act, 1.0, 0.0, 2)
    torch.cuda.synchronize()


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("mode,c", [(0, 32), (2, 32), (0, 5), (2, 5)])
def test_pooling_fused_activation(ext, dtype, mode, c):
    """max / avg pooling with strict ReLU folded in (forward) and f'(y) folded into the
    backward gather == pooling followed by a separate ReLU."""
    torch.manual_seed(mode * 10 + c)
    dev = "cuda"
    n, h, w, k, s = 3, 9, 9, 3, 2
    oh = ow = (h - k + s - 1) // s + 1 if (h - k) % s else (h - k) // s + 1
    oh = ow = -(-(h - k) // s) + 1
    x = torch.randn(n, h, w, c, device=dev).to(dtype)
    out_f = torch.empty(n, oh, ow, c, device=dev, dtype=dtype)
    out_p = torch.empty_like(out_f)
    offs_f = torch.zeros(n, oh, ow, c, device=dev, dtype=torch.int32)
    offs_p = torch.zeros_like(offs_f)
    ext.pool_forward(x, out_f, offs_f, oh, ow, k, k, s, s, mode, None, 3)
    ext.pool_forward(x, out_p, offs_p, oh, ow, k, k, s, s, mode, None, 0)
    torch.cuda.synchronize()
    assert torch.equal(out_f, torch.relu(out_p)) and torch.equal(offs_f, offs_p)
    err = torch.randn(n, oh, ow, c, device=dev).to(dtype)
    ei_f = torch.empty_like(x)
    ei_p = torch.empty_like(x)
    ext.pool_backward(err, offs_f, ei_f, oh, ow, k, k, s, s, mode == 2, out_f, 3, None, 0)
    masked = (err.float() * (out_f.float() > 0)).to(dtype)
    ext.pool_backward(masked, offs_p, ei_p, oh, ow, k, k, s, s, mode == 2, None, 0, None, 0)
    torch.cuda.synchronize()
    assert _rel(ei_f.float(), ei_p.float()) < (1e-6 if dtype == torch.float32 else 1e-2)
    # producer-side derivative: err_input *= f'(pooling input) (tanh: f' = 1.14381894 - 0.388484177 y^2)
    ei_d = torch.empty_like(x)
    ext.pool_backward(err, offs_p, ei_d, oh, ow, k, k, s, s, mode == 2, None, 0, x, 1)
    torch.cuda.synchronize()
    ref = ei_p.float() * 0 + 0      # plain backward of the unmasked error, then the derivative
    ext.pool_backward(err, offs_p, ei_p, oh, ow, k, k, s, s, mode == 2, None, 0, None, 0)
    torch.cuda.synchronize()
    ref = ei_p.float() * (1.14381894 - 0.388484177 * x.float() ** 2)
    assert _rel(ei_d.float(), ref) < (1e-6 if dtype == torch.float32 else 1e-2)


@pytest.mark.parametrize("src_dt,dst_dt", [(torch.float32, torch.bfloat16),
                                           (torch.float32, torch.float32)])
def test_gather_minibatch_with_channel_padding(ext, src_dt, dst_dt):
    """Device-resident dataset → minibatch (+ labels) and, in the same launch, the
    channel-padded (3 → 8) copy the first conv layer's vector gather consumes."""
    torch.manual_seed(5)
    dev = "cuda"
    total, rows, count = 50, 12, 9
    data = torch.randn(total, 8, 8, 3, device=dev).to(src_dt)
    labels = torch.randint(0, 10, (total,), device=dev, dtype=torch.int32)
    idx = torch.randperm(total, device=dev)[:rows].to(torch.int32)
    hdr = torch.cat([torch.tensor([count, 2, 0, 0], device=dev, dtype=torch.int32), idx])
    dst = torch.full((rows, 8, 8, 3), float("nan"), device=dev, dtype=dst_dt)
    pad = torch.full((rows, 8, 8, 8), float("nan"), device=dev, dtype=dst_dt)
    ldst = torch.full((rows,), -7, device=dev, dtype=torch.int32)
    ext.gather_minibatch(data, labels, hdr, dst, ldst, pad, 3)
    torch.cuda.synchronize()
    ref = data[idx.long()].to(dst_dt)
    ref[count:] = 0
    assert torch.equal(dst, ref)
    assert torch.equal(pad[..., :3], ref) and float(pad[..., 3:].abs().sum()) == 0.0
    assert torch.equal(ldst[:count], labels[idx.long()][:count]) and bool((ldst[count:] == -1).all())
    # without the padded copy
    dst2 = torch.empty_like(dst)
    ext.gather_minibatch(data, labels, hdr, dst2, ldst, None, 0)
    torch.cuda.synchronize()
    assert torch.equal(dst2, ref)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_fc_small_forward_fused_evaluator(ext, dtype):
    """softmax FC + evaluator in one launch == fc_small_forward followed by evaluate_softmax."""
    torch.manual_seed(11)
    dev = "cuda"
    batch, valid, n_in, n_out = 50, 43, 256, 10
    x = torch.randn(batch, n_in, device=dev).to(dtype)
    w = torch.randn(n_out, n_in, device=dev) * 0.1
    b = torch.randn(n_out, device=dev)
    labels = torch.randint(0, n_out, (batch,), device=dev, dtype=torch.int32)
    labels[5] = -1                                        # ignored sample
    bp = torch.tensor([float(valid), 1.0 / valid], device=dev)

    def fresh():
        return dict(out=torch.empty(batch, n_out, device=dev),
                    mi=torch.zeros(batch, dtype=torch.int32, device=dev),
                    err=torch.full((batch, n_out), float("nan"), device=dev).to(dtype),
                    n_err=torch.zeros(2, dtype=torch.int32, device=dev),
                    conf=torch.zeros(n_out, n_out, dtype=torch.int32, device=dev),
                    mx=torch.zeros(1, device=dev))
    a, f = fresh(), fresh()
    ext.fc_small_forward(x, w, b, a["out"], a["mi"], batch, n_in, n_out, 0, True, [])
    ext.evaluate_softmax(a["out"], a["mi"], labels, a["err"], bp, a["n_err"], a["conf"], a["mx"])
    ext.fc_small_forward(x, w, b, f["out"], f["mi"], batch, n_in, n_out, 0, True,
                         [labels, f["err"], bp, f["n_err"], f["mx"], f["conf"]])
    torch.cuda.synchronize()
    assert torch.equal(a["out"], f["out"]) and torch.equal(a["mi"], f["mi"])
    assert torch.equal(a["n_err"], f["n_err"]) and torch.equal(a["conf"], f["conf"])
    assert torch.allclose(a["err"].float(), f["err"].float(), atol=1e-6 if dtype == torch.float32 else 1e-3)
    assert abs(float(a["mx"]) - float(f["mx"])) < 1e-3


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("c", [32, 5])
def test_lrn_backward_with_producer_derivative(ext, dtype, c):
    """LRN backward with the producer's strict-ReLU derivative folded in == LRN backward
    followed by a separate err *= (x > 0)."""
    torch.manual_seed(c)
    dev = "cuda"
    x = torch.relu(torch.randn(3, 7, 7, c, device=dev)).to(dtype)
    ey = torch.randn(3, 7, 7, c, device=dev).to(dtype)
    plain = torch.empty_like(x)
    fused = torch.empty_like(x)
    ext.lrn_backward(ey, x, plain, 3, 5e-5, 0.75, 1.0, 0)
    ext.lrn_backward(ey, x, fused, 3, 5e-5, 0.75, 1.0, 3)
    torch.cuda.synchronize()
    ref = plain.float() * (x.float() > 0)
    assert _rel(fused.float(), ref) < (1e-6 if dtype == torch.float32 else 1e-2)


@pytest.mark.parametrize("M,N,K", [(128, 256, 512), (100, 72, 384), (257, 1000, 4096)])
@pytest.mark.parametrize("out_dt", [torch.bfloat16, torch.float32])
def test_gemm_fp8_e4m3(ext, M, N, K, out_dt):
    """tcgen05 kind::f8f6f4 GEMM on per-tensor-scaled e4m3 operands: exact (up to fp32
    accumulation order) against the same quantised operands multiplied in fp32, and within
    fp8 tolerance of the unquantised product."""
    torch.manual_seed(M + N)
    dev = "cuda"
    a = torch.randn(M, K, device=dev)
    b = torch.randn(N, K, device=dev) / K ** 0.5
    bias = torch.randn(N, device=dev)
    qa = torch.empty(M, K, device=dev, dtype=torch.uint8)
    qb = torch.empty(N, K, device=dev, dtype=torch.uint8)
    amax = torch.zeros(2, device=dev)
    ext.fp8_absmax(a, amax[0:1])
    ext.fp8_absmax(b, amax[1:2])
    ext.fp8_quantize(a, qa, amax[0:1])
    ext.fp8_quantize(b, qb, amax[1:2])
    torch.cuda.synchronize()
    assert abs(float(amax[0]) - float(a.abs().max())) < 1e-6
    sa, sb = 448.0 / float(amax[0]), 448.0 / float(amax[1])
    # our quantiser == torch's e4m3 cast of the scaled tensor
    ref_qa = (a * sa).to(torch.float8_e4m3fn)
    assert torch.equal(qa.view(torch.float8_e4m3fn).float(), ref_qa.float())
    out = torch.full((M, N), float("nan"), device=dev, dtype=out_dt)
    r = ext.gemm_fp8(qa, qb, out, bias, 3, 1.0 / (sa * sb))
    assert r == 0
    torch.cuda.synchronize()
    fa = qa.view(torch.float8_e4m3fn).float()
    fb = qb.view(torch.float8_e4m3fn).float()
    ref_q = torch.relu(fa @ fb.t() / (sa * sb) + bias)
    assert _rel(out.float(), ref_q) < (1e-2 if out_dt == torch.bfloat16 else 1e-5)
    ref = torch.relu(a @ b.t() + bias)
    assert _rel(out.float(), ref) < 6e-2


@pytest.mark.parametrize("M,N,K,f32,act", [(256, 256, 64, False, 0), (1024, 1024, 512, False, 3),
                                           (768, 384, 200, False, 0), (512, 256, 128, True, 0),
                                           (2048, 4096, 1024, False, 0)])
def test_gemm_pair_2cta_persistent(ext, M, N, K, f32, act):
    """csrc/gemm_pair.cu (cta_group::2, persistent, TMEM double buffering, TMA store) vs fp32
    PyTorch, with the 2x-NaN out-of-bounds guard."""
    torch.manual_seed(M + N)
    dev = "cuda"
    a = torch.randn(M, K, device=dev).bfloat16()
    b = torch.randn(N, K, device=dev).bfloat16()
    bias = torch.randn(N, device=dev)
    big = torch.full((2 * M, N), float("nan"), device=dev,
                     dtype=torch.float32 if f32 else torch.bfloat16)
    assert ext.gemm_pair(a, b, big[:M], bias, act, 0.5) == 0
    torch.cuda.synchronize()
    ref = 0.5 * (a.float() @ b.float().t()) + bias
    if act == 3:
        ref = torch.relu(ref)
    assert _rel(big[:M], ref) < (1e-5 if f32 else 1e-2)
    l2 = ((big[:M].float() - ref).norm() / ref.norm()).item()
    assert l2 < (1e-6 if f32 else 4e-3)
    assert torch.isnan(big[M:]).all()


@pytest.mark.parametrize("batch,n_out,n_in", [(128, 512, 1024), (64, 1000, 768), (200, 256, 4104)])
def test_fc_wgrad_pair(ext, batch, n_out, n_in):
    """gradW[out][in] = err^T . x on the 2-CTA kernel (both operands MN-major, K = batch)."""
    torch.manual_seed(batch)
    dev = "cuda"
    err = torch.randn(batch, n_out, device=dev).bfloat16()
    x = torch.randn(batch, n_in, device=dev).bfloat16()
    big = torch.full((2 * n_out, n_in), float("nan"), device=dev)
    assert ext.fc_wgrad_pair(err, x, big[:n_out]) == 0
    torch.cuda.synchronize()
    ref = err.float().t() @ x.float()
    assert _rel(big[:n_out], ref) < 1e-5
    assert torch.isnan(big[n_out:]).all()
