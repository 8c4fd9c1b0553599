"""Per-kernel parity (GPU): every C-ABI op against the same op in PyTorch fp64 on the CPU
(the oracle for single ops is torch itself: F.conv2d / F.linear / max_pool / autograd).

Tolerances: integer results (argmax indices) bit-exact; fp32 CUDA-core kernels and the TF32X3
(fp32-grade) tensor-core kernels <= 2e-5 relative L2; single-pass TF32 <= 3e-3 (its own bound).
"""
import os
import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

PRECS = {"fp32": 0, "tf32x3": 1, "tf32": 2}
TOL = {"fp32": 2e-5, "tf32x3": 2e-5, "tf32": 3e-3}


def _ops():
    from b200np import ops
    return ops


def rel(a, b):
    a = a.detach().double().cpu()
    b = b.detach().double().cpu()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def rnd(*shape, seed=0, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(*shape, generator=g, dtype=torch.float64) * scale)


def nhwc(t):  # NCHW fp64 cpu -> NHWC fp32 cuda
    return t.permute(0, 2, 3, 1).contiguous().float().cuda()


def from_nhwc(t):
    return t.permute(0, 3, 1, 2)


# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("prec", ["fp32", "tf32x3", "tf32"])
@pytest.mark.parametrize("cin,r,cout,hw,n", [(1, 5, 64, 32, 3), (3, 5, 64, 16, 3), (1, 3, 32, 32, 3), (1, 5, 64, 128, 3),
                                             (1, 5, 64, 6, 1), (1, 5, 64, 64, 37)])
def test_conv_small_fwd_and_wgrad(prec, cin, r, cout, hw, n):
    """Stem convolutions: CUDA-core fp32 kernels, and the tcgen05 kernels of the 1-channel 5x5 stem in the
    TF32 modes (ragged last tile, K-blocks that straddle images, chunk counts below and above the cap)."""
    ops = _ops()
    from b200np import lib
    P = {"fp32": lib.PREC_FP32_SIMT, "tf32x3": lib.PREC_TF32X3, "tf32": lib.PREC_TF32}[prec]
    tc = prec != "fp32" and (cin, r, cout) == (1, 5, 64)
    tol_y, tol_g = (2e-6, 1e-5) if not tc else ((3e-6, 1e-5) if prec == "tf32x3" else (2e-3, 2e-3))
    x, w, b = rnd(n, cin, hw, hw, seed=1), rnd(cout, cin, r, r, seed=2, scale=0.2), rnd(cout, seed=3)
    w.requires_grad_(True), b.requires_grad_(True)
    ref = F.relu(F.conv2d(x, w, b, stride=2, padding=r // 2))
    y = ops.conv_small_fwd(x.float().cuda(), w.detach().float().cuda(), b.detach().float().cuda(), prec=P)
    assert rel(from_nhwc(y), ref) < tol_y
    dy = rnd(*ref.shape, seed=4) * (ref > 0)  # gradient w.r.t. the pre-activation
    pre = F.conv2d(x, w, b, stride=2, padding=r // 2)
    pre.backward(dy)
    dw, db = ops.conv_small_wgrad(x.float().cuda(), nhwc(dy), w.shape, P)
    assert rel(dw, w.grad) < tol_g
    assert rel(db, b.grad) < tol_g


@pytest.mark.parametrize("prec", ["fp32", "tf32x3", "tf32"])
@pytest.mark.parametrize("cin,cout,hw,n", [(64, 64, 16, 3), (64, 64, 4, 5), (64, 64, 2, 70), (64, 64, 64, 2), (64, 64, 32, 3), (32, 48, 16, 2), (48, 64, 8, 2)])
def test_conv_block_ops(prec, cin, cout, hw, n):
    """3x3 s2 / 3x3 s1 / fused skip projection: forward, data gradient (with ReLU mask), weight grad."""
    ops = _ops()
    P, tol = PRECS[prec], TOL[prec]
    if prec != "fp32" and (cin, cout) != (64, 64):
        tol = TOL["fp32"]  # these shapes route to the CUDA-core kernels in every mode
    x = rnd(n, cin, hw, hw, seed=1).abs()
    w1, b1 = rnd(cout, cin, 3, 3, seed=2, scale=0.05).requires_grad_(), rnd(cout, seed=3, scale=0.1).requires_grad_()
    x.requires_grad_(True)
    # --- conv 3x3 stride 2 + ReLU
    pre1 = F.conv2d(x, w1, b1, stride=2, padding=1)
    h = F.relu(pre1)
    xg = nhwc(x.detach())
    p1 = ops.pack_conv_weight(w1.detach().float().cuda())
    hg = ops.conv_fwd(xg, p1, b1.detach().float().cuda(), 2, 1, P)
    assert rel(from_nhwc(hg), h) < tol
    if hw < 4:
        return
    if cin == cout:
        # --- conv 3x3 stride 1 + 1x1 stride-2 skip projection + add + ReLU (one launch)
        w2, b2 = rnd(cout, cout, 3, 3, seed=4, scale=0.05).requires_grad_(), rnd(cout, seed=5, scale=0.1).requires_grad_()
        ws, bs = rnd(cout, cin, 1, 1, seed=6, scale=0.1).requires_grad_(), rnd(cout, seed=7, scale=0.1).requires_grad_()
        y = F.relu(F.conv2d(h, w2, b2, padding=1) + F.conv2d(x, ws, bs, stride=2))
        p2 = ops.pack_conv_weight(w2.detach().float().cuda())
        ps = ops.pack_conv_weight(ws.detach().float().cuda())
        hgx = nhwc(h.detach())
        yg = ops.conv_fwd(hgx, p2, b2.detach().float().cuda(), 1, 1, P,
                          skip=(xg, ps, bs.detach().float().cuda(), 2))
        assert rel(from_nhwc(yg), y) < tol
        gy = rnd(*y.shape, seed=8)
        y.backward(gy)
        dz = (gy * (y > 0)).detach()        # gradient at the pre-activation of the block output
        dzg = nhwc(dz)
        dw2, db2, _ = ops.conv_wgrad(hgx, dzg, 3, 1, P)
        dws, _, _ = ops.conv_wgrad(xg, dzg, 1, 2, P, want_db=False)
        assert rel(dw2, w2.grad) < tol and rel(db2, b2.grad) < 1e-5 and rel(dws, ws.grad) < tol
        if prec != "fp32":   # fused: the skip projection's gradient as an extra tap of conv2's weight gradient
            dw2f, db2f, dwsf = ops.conv_wgrad(hgx, dzg, 3, 1, P, skip=(xg, 2))
            assert rel(dw2f, w2.grad) < tol and rel(db2f, b2.grad) < 1e-5 and rel(dwsf, ws.grad) < tol
        dh = ops.conv_dgrad(dzg, p2, hgx.shape, 1, P, mask_src=hgx)
        # reference dh: gradient at conv1's pre-activation
        hh = h.detach().requires_grad_()
        F.conv2d(hh, w2.detach(), None, padding=1).backward(dz)
        dh_ref = hh.grad * (h > 0)
        assert rel(from_nhwc(dh), dh_ref) < tol
        dw1, db1, _ = ops.conv_wgrad(xg, dh, 3, 2, P)
        assert rel(dw1, w1.grad) < tol and rel(db1, b1.grad) < max(tol, 2e-5)
        dx = ops.conv_dgrad(dh, p1, xg.shape, 2, P, mask_src=xg, skip=(dzg, ps, 2))
        assert rel(from_nhwc(dx), x.grad * (x > 0)) < tol
    else:
        gy = rnd(*h.shape, seed=8)
        h.backward(gy)
        dz = nhwc((gy * (h > 0)).detach())
        dw1, db1, _ = ops.conv_wgrad(xg, dz, 3, 2, P)
        assert rel(dw1, w1.grad) < tol and rel(db1, b1.grad) < max(tol, 2e-5)
        dx = ops.conv_dgrad(dz, p1, xg.shape, 2, P, mask_src=None)
        assert rel(from_nhwc(dx), x.grad) < tol


def test_pools_and_flatten():
    ops = _ops()
    x = rnd(5, 64, 4, 4, seed=1)
    x[0, :, :, :] = 0.0          # all-equal window: first index wins (SURVEY.md 2.1 L3)
    x[1, 3, 0, 0] = x[1, 3, 0, 1] = 7.0   # tie inside a window
    x = F.relu(x).requires_grad_()
    ref, idx = F.adaptive_max_pool2d(x, (2, 2), return_indices=True)
    xg = nhwc(x.detach())
    out, gi = ops.amp2_flatten_fwd(xg)
    assert torch.equal(out.cpu().double(), ref.reshape(5, -1).double().float().double())
    assert torch.equal(gi.cpu().long(), idx.reshape(5, -1))
    g = rnd(5, 256, seed=2)
    ref.reshape(5, -1).backward(g)
    dx = ops.amp2_flatten_bwd(g.float().cuda(), gi, xg, torch.empty_like(xg))
    assert rel(from_nhwc(dx), x.grad * (x > 0)) < 1e-6
    # reshape path
    x2 = rnd(3, 64, 2, 2, seed=3)
    flat = ops.nhwc_to_nchw_flat(nhwc(x2))
    assert torch.equal(flat.cpu(), x2.reshape(3, -1).float())
    back = ops.nchw_flat_to_nhwc(flat, None, torch.empty(3, 2, 2, 64, device="cuda"), mask=False)
    assert torch.equal(from_nhwc(back).cpu(), x2.float())
    # MaxPool2d(2,2): 48 channels take the 16-byte kernels, 6 channels the scalar ones
    for Cp in (48, 6):
        x3 = F.relu(rnd(2, Cp, 8, 8, seed=4))
        x3[0, 0, 0:2, 0:2] = 1.5
        x3.requires_grad_()
        ref3, idx3 = F.max_pool2d(x3, 2, return_indices=True)
        y3, i3 = ops.maxpool2x2_fwd(nhwc(x3.detach()))
        assert torch.equal(from_nhwc(y3).cpu(), ref3.float())
        iy, ix = idx3 // 8, idx3 % 8
        assert torch.equal(from_nhwc(i3).cpu().long(), (iy % 2) * 2 + ix % 2)
        g3 = rnd(*ref3.shape, seed=5)
        ref3.backward(g3)
        d3 = ops.maxpool2x2_bwd(nhwc(g3), i3, nhwc(x3.detach()))
        assert rel(from_nhwc(d3), x3.grad * (x3 > 0)) < 1e-6


@pytest.mark.parametrize("prec", ["fp32", "tf32x3", "tf32"])
@pytest.mark.parametrize("M,N,K", [(420, 256, 272), (37, 2, 256), (300, 100, 80), (1000, 1419, 256), (5, 16, 2),
                                   (3360, 256, 1419)])
def test_gemm_forward_roles(M, N, K, prec):
    """All three autograd roles of a dense layer (K-major / MN-major operand combinations), K and N tails,
    the fused epilogue -- on the CUDA-core kernel (fp32) and the tcgen05 kernel (tf32x3 / tf32)."""
    ops = _ops()
    P = PRECS[prec]
    t6 = {"fp32": 2e-6, "tf32x3": 4e-6, "tf32": 3e-3}[prec]
    x, w, b = rnd(M, K, seed=1), rnd(N, K, seed=2, scale=0.1), rnd(N, seed=3)
    xg, wg, bg = x.float().cuda(), w.float().cuda(), b.float().cuda()
    y = torch.empty(M, N, device="cuda")
    ops.gemm(xg.data_ptr(), wg.data_ptr(), y.data_ptr(), M, N, K, K, 1, 1, K, N, bias=bg.data_ptr(), act=1, prec=P)
    assert rel(y, F.relu(F.linear(x, w, b))) < t6
    dz = rnd(M, N, seed=4)
    dzg = dz.float().cuda()
    dx = torch.empty(M, K, device="cuda")
    ops.gemm(dzg.data_ptr(), wg.data_ptr(), dx.data_ptr(), M, K, N, N, 1, K, 1, K, prec=P)
    assert rel(dx, dz @ w) < t6
    dw = torch.empty(N, K, device="cuda")
    ops.gemm(dzg.data_ptr(), xg.data_ptr(), dw.data_ptr(), N, K, M, 1, N, K, 1, K, prec=P)
    assert rel(dw, dz.t() @ x) < t6
    db = ops.colsum(dzg, M, N, N)
    assert rel(db, dz.sum(0)) < 2e-6
    # beta / tanh / row_scale*addend epilogue
    add, rs = rnd(M, N, seed=5), rnd(M, seed=6)
    y2 = y.clone()
    ops.gemm(xg.data_ptr(), wg.data_ptr(), y2.data_ptr(), M, N, K, K, 1, 1, K, N, alpha=0.5, beta=1.0, act=2,
             row_scale=rs.float().cuda(), addend=add.float().cuda(), ld_add=N, prec=P)
    ref2 = torch.tanh(0.5 * (x @ w.t()) + F.relu(F.linear(x, w, b)) + rs[:, None] * add)
    assert rel(y2, ref2) < 3 * t6


@pytest.mark.parametrize("prec", ["fp32", "tf32x3"])
def test_gemm_grouped_heads(prec):
    ops = _ops()
    rows, K, d, H = 45, 256, 256, 8
    x = rnd(rows, K, seed=1)
    ws = [rnd(d, K, seed=10 + h, scale=0.06) for h in range(H)]
    bs = [rnd(d, seed=20 + h) for h in range(H)]
    xg = x.float().cuda()
    wg = [w.float().cuda() for w in ws]
    bg = [b.float().cuda() for b in bs]
    y = torch.empty(rows, H * d, device="cuda")
    ops.gemm([xg.data_ptr()] * H, [w.data_ptr() for w in wg], [y.data_ptr() + 4 * h * d for h in range(H)],
             rows, d, K, K, 1, 1, K, H * d, bias=[b.data_ptr() for b in bg], prec=PRECS[prec])
    ref = torch.cat([F.linear(x, w, b) for w, b in zip(ws, bs)], dim=1)
    assert rel(y, ref) < 4e-6


def test_elementwise_and_reductions():
    ops = _ops()
    x = rnd(1000, 37, seed=1).float().cuda()
    y = F.relu(rnd(1000, 37, seed=2)).float().cuda()
    assert torch.equal(ops.act_bwd(x, y, 1), x * (y > 0))
    t = torch.tanh(rnd(1000, 37, seed=3)).float().cuda()
    assert rel(ops.act_bwd(x, t, 2), x.double().cpu() * (1 - t.double().cpu() ** 2)) < 1e-6
    r = ops.repeat_rows(x[:10].contiguous(), 7)
    assert torch.equal(r, x[:10].repeat_interleave(7, dim=0))
    assert rel(ops.repeat_rows_bwd(r, 7), 7 * x[:10].double().cpu()) < 1e-6
    assert float(ops.reduce(x.view(-1), 0)) == float(x.max())
    assert abs(float(ops.reduce(x.view(-1), 1)) - float(x.double().sum())) < 1e-2
    z = ops.zeros((5, 3), x)
    assert float(z.abs().sum()) == 0.0
    ops.axpy(z, torch.ones(5, 3, device="cuda"), 2.5)
    assert float(z.sum()) == 37.5
    s = torch.tensor([3.0], device="cuda")
    assert torch.equal(ops.scale_by_device_scalar(x, s), 3.0 * x)


@pytest.mark.parametrize("mode", [0, 1])
def test_ctx_aggregate(mode):
    ops = _ops()
    f = F.relu(rnd(6, 15, 256, seed=1))
    f[:, :, :40] = 0.0            # post-ReLU ties at zero are common: FIRST index must win
    f[2, 3, 50] = f[2, 9, 50] = 9.0
    f.requires_grad_()
    fg = f.detach().float().cuda()
    out, idx = ops.ctx_aggregate_fwd(fg, mode)
    if mode == 0:
        ref = f.mean(1)
        assert rel(out, ref) < 1e-6
    else:
        ref, ridx = f.max(1)
        assert torch.equal(out.cpu(), ref.float())
        assert torch.equal(idx.cpu().long(), ridx)
    g = rnd(6, 256, seed=2)
    ref.backward(g)
    df = ops.ctx_aggregate_bwd(g.float().cuda(), idx, 6, 15, 256, mode)
    assert rel(df, f.grad) < 1e-6


@pytest.mark.parametrize("task,kind", [("distractor", 0), ("shapenet_3d", 1), ("shapenet_1d", 2)])
def test_losses_against_reference_golden(task, kind, golden):
    ops = _ops()
    mu = torch.from_numpy(golden[f"loss/{task}/mu"]).cuda()
    y = torch.from_numpy(golden[f"loss/{task}/y"]).cuda()
    loss, dmu = ops.loss_fwd_bwd(mu.contiguous(), y.contiguous(), kind)
    ref = float(golden[f"loss/{task}/loss"])
    assert abs(float(loss) - ref) < 2e-6 * abs(ref)
    assert rel(dmu, torch.from_numpy(golden[f"loss/{task}/dmu"])) < 2e-6
    if task == "shapenet_1d":
        lt, _ = ops.loss_fwd_bwd(mu.contiguous(), y.contiguous(), 3, want_grad=False)
        ref_t = float(golden[f"loss/{task}/loss_test"])
        assert abs(float(lt) - ref_t) < 1e-4 * abs(ref_t)


@pytest.mark.parametrize("kind", [0, 2])
@pytest.mark.parametrize("R,L", [(40000, 2), (40001, 2), (33333, 3), (3_000_001, 2)])
def test_loss_large_batches(kind, R, L):
    """Beyond 16384 rows the loss runs multi-block (last-block reduction); two-wide labels take the 16-byte form with an
    odd tail row, wider labels the scalar-row form.  Reference: trainer/losses.py:35-36 (distractor), :59-61 (azimuth)."""
    ops = _ops()
    mu = rnd(R, 2, seed=5).float().cuda()
    y = rnd(R, L, seed=6).float().cuda()
    for _ in range(2):  # the ticket counter must be re-armed by the first call
        loss, dmu = ops.loss_fwd_bwd(mu, y, kind)
    m64 = mu.double().requires_grad_()
    e = y[:, :2].double() - m64
    ref = e.norm(dim=1).mean() if kind == 0 else (e * e).sum(1).mean()
    ref.backward()
    assert abs(float(loss) - float(ref)) < 2e-6 * abs(float(ref))
    assert rel(dmu, m64.grad) < 1e-6
    lo, none = ops.loss_fwd_bwd(mu, y, kind, want_grad=False)
    assert none is None and abs(float(lo) - float(ref)) < 2e-6 * abs(float(ref))


def test_adam_matches_torch():
    ops = _ops()
    n = 10007
    p0, gs = rnd(n, seed=1).float(), [rnd(n, seed=10 + i).float() for i in range(3)]
    p_ref = p0.clone().requires_grad_()
    opt = torch.optim.Adam([p_ref], lr=1e-3)
    p, m, v = p0.clone().cuda(), torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")
    for i, g in enumerate(gs):
        p_ref.grad = g.clone()
        opt.step()
        ops.adam_step(p, g.cuda(), m, v, n, 1e-3, 0.9, 0.999, 1e-8, 0.0, i + 1)
    assert rel(p, p_ref) < 1e-6


@pytest.mark.parametrize("prec", ["fp32", "tf32x3"])
@pytest.mark.parametrize("T,H,nt,nc,d", [(2, 8, 5, 4, 64), (2, 8, 21, 15, 256), (1, 2, 36, 25, 64)])
def test_favor_attention_fwd_bwd(prec, T, H, nt, nc, d):
    """Fused FAVOR+ (re-associated) vs the closed-form fp64 restatement of the reference
    (oracle.np_oracle.favor_attention_fwd_bwd, itself checked against autograd through the
    reference formulation in tests/test_oracle_golden.py)."""
    from b200np.engine import FavorAttentionFn
    from oracle import np_oracle
    M = int(d * np.log(d))
    xq, xk, v = rnd(T, nt, H, d, seed=1), rnd(T, nc, H, d, seed=2), rnd(T, nc, H, d, seed=3)
    if nc >= 4:
        xk[0, 1] = xk[0, 0]  # duplicated context row -> exact tie of the global key max candidates
    P = rnd(M, d, seed=4)
    d_out = rnd(T, H, nt, d, seed=5)
    to_bh = lambda t: t.permute(0, 2, 1, 3)  # [T,n,H,d] -> [T,H,n,d]
    out_ref, (dq_ref, dk_ref, dv_ref) = np_oracle.favor_attention_fwd_bwd(to_bh(xq), to_bh(xk), to_bh(v), P, d_out)
    q_g = xq.reshape(T * nt, H * d).float().cuda().requires_grad_()
    k_g = xk.reshape(T * nc, H * d).float().cuda().requires_grad_()
    v_g = v.reshape(T * nc, H * d).float().cuda().requires_grad_()
    out = FavorAttentionFn.apply(PRECS[prec], T, H, nt, nc, q_g, k_g, v_g, P.float().cuda())
    # out [T*nt, d*H] with index e*H + h
    out_bh = out.view(T, nt, d, H).permute(0, 3, 1, 2)
    assert rel(out_bh, out_ref) < 2e-5
    out.backward(d_out.permute(0, 2, 3, 1).reshape(T * nt, d * H).float().cuda())
    from_rows = lambda g, n: g.view(T, n, H, d).permute(0, 2, 1, 3)
    # calibration (tools/diag_precision.py, d=256): the reference formulation itself in fp32 is off by
    # 1e-3 (CPU) .. 6e-3 (GPU) on dq and 1e-5 on dk (row-argmax / global-max routing of tiny terms)
    assert rel(from_rows(v_g.grad, nc), dv_ref) < 2e-5
    assert rel(from_rows(k_g.grad, nc), dk_ref) < 2e-3
    assert rel(from_rows(q_g.grad, nt), dq_ref) < 2e-2


@pytest.mark.parametrize("prec", ["fp32", "tf32x3", "tf32"])
@pytest.mark.parametrize("rows,H,d,K", [(300, 8, 256, 256), (37, 3, 64, 96)])
def test_gemm_sum_groups(prec, rows, H, d, K):
    """dX = sum_h dY[:, h*d:(h+1)*d] @ W_h (the per-head AttnLinear data gradient, ANPDistractor.py:83-96) as ONE
    product whose K dimension runs over the groups."""
    ops = _ops()
    from b200np import lib
    P = {"fp32": lib.PREC_FP32_SIMT, "tf32x3": lib.PREC_TF32X3, "tf32": lib.PREC_TF32}[prec]
    dy = rnd(rows, H * d, seed=11)
    ws = [rnd(d, K, seed=20 + h, scale=0.1) for h in range(H)]
    ref = sum(dy[:, h * d:(h + 1) * d] @ ws[h] for h in range(H))
    dyc = dy.float().cuda()
    wc = [w.float().cuda() for w in ws]
    dx = torch.full((rows, K), float("nan"), device="cuda")
    ops.gemm([dyc.data_ptr() + 4 * h * d for h in range(H)], [w.data_ptr() for w in wc], [dx.data_ptr()] * H,
             rows, K, d, H * d, 1, K, 1, K, prec=P, sum_groups=True)
    assert rel(dx, ref) < (2e-3 if prec == "tf32" else 3e-6)


def _pack_bits(act_nhwc):
    """[N,H,W,64] -> int32 [N,H,W,2]: bit j of word h = (act[..., 32h + j] > 0) (include/b200np.h)."""
    g = (act_nhwc > 0).to(torch.int64).reshape(*act_nhwc.shape[:-1], 2, 32)
    w = (g << torch.arange(32, device=g.device, dtype=torch.int64)).sum(-1)
    return torch.where(w >= 2 ** 31, w - 2 ** 32, w).to(torch.int32).contiguous()


@pytest.mark.parametrize("prec", ["tf32x3", "tf32"])
def test_stem_relu_bits(prec):
    """The tcgen05 stem writes the ReLU gates of its output as 1 bit per element."""
    ops = _ops()
    from b200np import lib
    P = {"tf32x3": lib.PREC_TF32X3, "tf32": lib.PREC_TF32}[prec]
    x, w, b = rnd(5, 1, 64, 64, seed=1).float().cuda(), rnd(64, 1, 5, 5, seed=2, scale=0.2).float().cuda(), rnd(64, seed=3).float().cuda()
    bits = torch.full((5, 32, 32, 2), 0x5a5a5a5a, device="cuda", dtype=torch.int32)
    y = ops.conv_small_fwd(x, w, b, prec=P, relu_bits=bits)
    assert torch.equal(bits, _pack_bits(y))
    assert 0.2 < float((y > 0).float().mean()) < 0.8


@pytest.mark.parametrize("prec", ["fp32", "tf32x3"])
@pytest.mark.parametrize("hw,n,stride", [(64, 2, 2), (32, 3, 1), (8, 4, 2), (8, 4, 1)])
def test_conv_dgrad_mask_bits_equals_float_mask(prec, hw, n, stride):
    """The packed gates give bit-identical data gradients to the float activation mask on every kernel path
    (halo incl. the fused stride-2 classes, gather, CUDA cores)."""
    ops = _ops()
    from b200np import lib
    P = {"fp32": lib.PREC_FP32_SIMT, "tf32x3": lib.PREC_TF32X3}[prec]
    w = rnd(64, 64, 3, 3, seed=5, scale=0.05).float().cuda()
    ws = rnd(64, 64, 1, 1, seed=6, scale=0.1).float().cuda()
    pw, pws = ops.pack_conv_weight(w), ops.pack_conv_weight(ws)
    act = rnd(n, hw, hw, 64, seed=7).float().cuda()                       # NHWC activation whose sign gates dx
    dy = rnd(n, hw // stride, hw // stride, 64, seed=8).float().cuda()
    skip = (rnd(n, hw // stride, hw // stride, 64, seed=9).float().cuda(), pws, 2) if stride == 2 else None
    a = ops.conv_dgrad(dy, pw, act.shape, stride, P, mask_src=act, skip=skip)
    b = ops.conv_dgrad(dy, pw, act.shape, stride, P, mask_src=None, skip=skip, mask_bits=_pack_bits(act))
    assert torch.equal(a, b)
    assert float((a == 0).float().mean()) > 0.3


def test_baco_aggregation():
    """Bayesian context aggregation forward/backward against torch fp64 autograd (CNPDistractor.py:60-75)."""
    ops = _ops()
    T, nc, D = 3, 7, 256
    mu = rnd(T, nc, D, seed=1).requires_grad_(True)
    s = (rnd(T, nc, D, seed=2) * 3).requires_grad_(True)      # covers softplus' linear branch (> 20 is rare: add one)
    with torch.no_grad():
        s[0, 0, 0] = 25.0
    var = 1e-5 + F.softplus(s)
    sig_inv = 1.0 / var
    sz = 1.0 / (1.0 + sig_inv.sum(1))
    ref = sz * (sig_inv * mu).sum(1)
    dr = rnd(T, D, seed=3)
    ref.backward(dr)
    r = ops.baco_fwd(mu.detach().float().cuda(), s.detach().float().cuda())
    assert rel(r, ref) < 2e-6
    dmu, ds = ops.baco_bwd(dr.float().cuda(), mu.detach().float().cuda(), s.detach().float().cuda(), r)
    assert rel(dmu, mu.grad) < 5e-6
    assert rel(ds, s.grad) < 5e-6


@pytest.mark.parametrize("hw,n,stride,skip", [(64, 2, 1, True), (64, 2, 2, False), (8, 5, 1, True), (8, 5, 2, False)])
def test_conv_fwd_relu_bits(hw, n, stride, skip):
    """The tensor-core forward kernels (halo and gather paths) emit the gates of their ReLU output as packed bits."""
    ops = _ops()
    from b200np import lib
    w = rnd(64, 64, 3, 3, seed=5, scale=0.05).float().cuda()
    ws = rnd(64, 64, 1, 1, seed=6, scale=0.1).float().cuda()
    b = rnd(64, seed=7, scale=0.1).float().cuda()
    x = rnd(n, hw, hw, 64, seed=8).float().cuda()
    xs = rnd(n, 2 * hw // stride, 2 * hw // stride, 64, seed=9).float().cuda()
    sk = (xs, ops.pack_conv_weight(ws), b, 2) if skip else None
    y, bits = ops.conv_fwd(x, ops.pack_conv_weight(w), b, stride, lib.ACT_RELU, lib.PREC_TF32X3, skip=sk, want_bits=True)
    assert bits is not None and torch.equal(bits, _pack_bits(y))
    assert 0.2 < float((y > 0).float().mean()) < 0.8


_FAVOR_CHILD = r"""
import sys, numpy as np, torch
sys.path[:0] = [sys.argv[1], sys.argv[2]]
from b200np import lib
from b200np.engine import FavorAttentionFn
T, H, nt, nc, d = 2, 8, 21, 15, 256
M = int(d * np.log(d))
g = torch.Generator().manual_seed(1)
r = lambda *s: torch.randn(*s, generator=g)
xq, xk, v, P, do = r(T * nt, H * d), r(T * nc, H * d), r(T * nc, H * d), r(M, d), r(T * nt, d * H)
q_g, k_g, v_g = (t.cuda().requires_grad_() for t in (xq, xk, v))
out = FavorAttentionFn.apply(lib.PREC_TF32X3, T, H, nt, nc, q_g, k_g, v_g, P.cuda())
out.backward(do.cuda())
np.savez(sys.argv[3], out=out.detach().cpu().numpy(), dq=q_g.grad.cpu().numpy(), dk=k_g.grad.cpu().numpy(), dv=v_g.grad.cpu().numpy())
"""


def test_favor_cluster_split_variants_agree(tmp_path):
    """B200NP_FAVOR_SPLIT = 1 | 2 | 4 | 8 CTAs per (task, head) (thread-block cluster, DSMEM reduction in rank order): the
    forward tile is the same sum in a different association, so outputs and gradients agree to fp32 rounding."""
    import subprocess
    import sys
    from conftest import PKG, ROOT
    res = {}
    for S in (1, 2, 4, 8):
        path = str(tmp_path / f"favor_{S}.npz")
        env = dict(os.environ, B200NP_FAVOR_SPLIT=str(S))
        r = subprocess.run([sys.executable, "-c", _FAVOR_CHILD, ROOT, PKG, path], capture_output=True, text=True, env=env,
                           timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        res[S] = np.load(path)
    bad = []
    for S in (2, 4, 8):
        for k, tol in (("out", 2e-6), ("dv", 2e-6), ("dk", 2e-5), ("dq", 2e-3)):
            # dq / dk route tiny terms through the row / global arg-max: the reference formulation itself moves by 1e-3
            # (dq) and 1e-5 (dk) between fp32 implementations (tools/diag_precision.py), so a re-associated fp32 sum does too
            a, b = res[S][k].astype(np.float64), res[1][k].astype(np.float64)
            e = np.linalg.norm(a - b) / np.linalg.norm(b)
            print(f"split {S} vs 1: {k} {e:.2e}")
            if not e <= tol:
                bad.append((S, k, e))
    assert not bad, bad


@pytest.mark.parametrize("prec", ["tf32x3", "tf32"])
@pytest.mark.parametrize("N,H,Cin,Cout", [(3, 16, 32, 48), (2, 32, 48, 64), (5, 16, 8, 64), (70, 16, 32, 48)])
def test_implicit_conv_gemm(prec, N, H, Cin, Cout):
    """b200np_gemm with a VIRTUAL tap-major im2col operand (conv_operand): forward (A virtual), weight gradient (B virtual)
    and the tap-major col2im, against F.conv2d and its autograd (3x3, stride 2, padding 1)."""
    ops = _ops()
    P = PRECS[prec]
    x = rnd(N, Cin, H, H, seed=1)
    w = rnd(Cout, Cin, 3, 3, seed=2, scale=0.2)
    b = rnd(Cout, seed=3)
    dy = rnd(N, Cout, H // 2, H // 2, seed=4)
    xr, wr = x.clone().requires_grad_(), w.clone().requires_grad_()
    y_ref = F.conv2d(xr, wr, b, stride=2, padding=1)
    y_ref.backward(dy)
    xg, dyg = nhwc(x), nhwc(dy)
    wt = ops.conv_weight_tapmajor(w.float().cuda())
    assert torch.equal(ops.conv_weight_tapmajor(wt, to_tapmajor=False).cpu(), w.float())
    M, K = N * (H // 2) ** 2, 9 * Cin
    y = torch.full((N, H // 2, H // 2, Cout), float("nan"), device="cuda")
    ops.gemm(xg.data_ptr(), wt.data_ptr(), y.data_ptr(), M, Cout, K, K, 1, 1, K, Cout, bias=b.float().cuda().data_ptr(),
             prec=P, conv=(1, H, H, Cin))
    assert rel(y.permute(0, 3, 1, 2), y_ref) < TOL[prec]
    dwt = torch.full((Cout, K), float("nan"), device="cuda")
    ops.gemm(dyg.data_ptr(), xg.data_ptr(), dwt.data_ptr(), Cout, K, M, 1, Cout, K, 1, K, prec=P, conv=(2, H, H, Cin))
    assert rel(ops.conv_weight_tapmajor(dwt, to_tapmajor=False), wr.grad) < TOL[prec]
    dcol = torch.empty(M, K, device="cuda")
    ops.gemm(dyg.data_ptr(), wt.data_ptr(), dcol.data_ptr(), M, K, Cout, Cout, 1, K, 1, K, prec=P)
    dx = ops.col2im3x3s2_tapmajor(dcol, tuple(xg.shape))
    assert rel(dx.permute(0, 3, 1, 2), xr.grad) < TOL[prec]
    gate = (x > 0).float()
    dxm = ops.col2im3x3s2_tapmajor(dcol, tuple(xg.shape), mask=nhwc(x))
    assert rel(dxm.permute(0, 3, 1, 2), xr.grad * gate) < TOL[prec]


def test_implicit_conv_gemm_refuses_what_it_cannot_do():
    """The implicit convolution exists on the tensor-core path only: fp32 mode, a channel count that is not a multiple of
    four or a product too small for a tile raise instead of silently taking another route."""
    ops = _ops()
    from b200np import lib
    x = torch.zeros(2, 8, 8, 8, device="cuda")
    wt = torch.zeros(16, 72, device="cuda")
    y = torch.zeros(2, 4, 4, 16, device="cuda")
    for prec, conv in ((lib.PREC_FP32_SIMT, (1, 8, 8, 8)), (lib.PREC_TF32X3, (1, 8, 8, 6)), (lib.PREC_TF32X3, (1, 8, 8, 8))):
        with pytest.raises(lib.B200NPError):
            ops.gemm(x.data_ptr(), wt.data_ptr(), y.data_ptr(), 32, 16, 72, 72, 1, 1, 72, 16, prec=prec, conv=conv)


@pytest.mark.parametrize("Cin,R,Cout", [(3, 5, 64), (1, 3, 32)])
def test_small_cin_im2col_gemm_stem(Cin, R, Cout):
    """b200np_im2col_small + b200np_gemm = the stride-2 stem convolution and its weight gradient (used where the tcgen05
    stem kernel does not apply: 3-channel images), against F.conv2d."""
    ops = _ops()
    from b200np import lib
    N, H = 6, 32
    x, w, b = rnd(N, Cin, H, H, seed=1), rnd(Cout, Cin, R, R, seed=2, scale=0.2), rnd(Cout, seed=3)
    dy = rnd(N, Cout, H // 2, H // 2, seed=4)
    wr = w.clone().requires_grad_()
    y_ref = F.conv2d(x, wr, b, stride=2, padding=R // 2)
    y_ref.backward(dy)
    col = ops.im2col_small(x.float().cuda(), R, R // 2)
    K, M = Cin * R * R, N * (H // 2) ** 2
    ref_col = F.unfold(x, R, padding=R // 2, stride=2).permute(0, 2, 1).reshape(M, K)
    assert col.shape == (M, (K + 3) // 4 * 4)
    assert torch.equal(col[:, :K].cpu(), ref_col.float()) and float(col[:, K:].abs().sum()) == 0.0
    if K >= 32:   # the tensor-core GEMM needs one full K-block; thinner stems stay on the direct kernels
        wc = w.float().cuda().contiguous()
        y = torch.empty(M, Cout, device="cuda")
        ops.gemm(col.data_ptr(), wc.data_ptr(), y.data_ptr(), M, Cout, K, col.shape[1], 1, 1, K, Cout,
                 bias=b.float().cuda().data_ptr(), prec=lib.PREC_TF32X3)
        assert rel(y.view(N, H // 2, H // 2, Cout).permute(0, 3, 1, 2), y_ref) < 2e-5
        dyg = nhwc(dy)
        dw = torch.empty(Cout, K, device="cuda")
        ops.gemm(dyg.data_ptr(), col.data_ptr(), dw.data_ptr(), Cout, K, M, 1, Cout, col.shape[1], 1, K, prec=lib.PREC_TF32X3)
        assert rel(dw.view_as(wc), wr.grad) < 2e-5
