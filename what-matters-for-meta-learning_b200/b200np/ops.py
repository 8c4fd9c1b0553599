"""Tensor-level wrappers over the C ABI: argument checking, output allocation (torch is used for
device memory and streams only), and the call into libb200np.so on torch's current stream."""
import ctypes as C

import torch

from . import lib
from .lib import LIB, GemmDesc, check

F32 = torch.float32


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return C.c_void_p(0 if t is None else t.data_ptr())


def _chk(t, name):
    if t is None:
        return
    if not t.is_cuda:
        raise lib.B200NPError(f"{name}: tensor is on {t.device}; the B200 path has no CPU fallback")
    if t.dtype != F32 and t.dtype not in (torch.int32, torch.int8):
        raise lib.B200NPError(f"{name}: dtype {t.dtype} unsupported")
    if not t.is_contiguous():
        raise lib.B200NPError(f"{name}: tensor must be contiguous")


def empty(shape, like, dtype=F32):
    return torch.empty(shape, device=like.device, dtype=dtype)


# ----------------------------------------------------------------------------------------------
# convolutions
# ----------------------------------------------------------------------------------------------
def relu_bits_supported(Cin, R, Cout, prec):
    """The tcgen05 stem kernel can emit the packed ReLU gates (include/b200np.h)."""
    return prec != lib.PREC_FP32_SIMT and (Cin, R, Cout) == (1, 5, 64)


def conv_small_fwd(x, w, b, out=None, relu=True, prec=lib.PREC_FP32_SIMT, relu_bits=None):
    """x NCHW [N,Cin,H,W] -> NHWC [N,H/2,W/2,Cout] (stride 2, pad R//2).  relu_bits: optional int32 tensor
    [N,H/2,W/2,2] receiving the ReLU gates, 1 bit per element."""
    for t, n in ((x, "x"), (w, "w"), (b, "b"), (out, "out")):
        _chk(t, n)
    N, Cin, H, W = x.shape
    Cout, _, R, _ = w.shape
    if out is None:
        out = empty((N, H // 2, W // 2, Cout), x)
    check(LIB.b200np_conv_small_fwd(_ptr(x), _ptr(w), _ptr(b), _ptr(out), N, Cin, H, W, Cout, R, 2, R // 2,
                                    int(relu), prec, _ptr(relu_bits), _stream()), "conv_small_fwd")
    return out


def conv_small_wgrad(x, dy, w_shape, prec=lib.PREC_FP32_SIMT):
    N, Cin, H, W = x.shape
    Cout, _, R, _ = w_shape
    _chk(x, "x"), _chk(dy, "dy")
    ws_bytes = LIB.b200np_conv_small_wgrad_workspace(N, Cin, H, W, Cout, R, 2, R // 2, prec)
    ws = torch.empty(max(ws_bytes // 4, 1), device=x.device, dtype=F32)
    dw = empty(tuple(w_shape), x)
    db = empty((Cout,), x)
    check(LIB.b200np_conv_small_wgrad(_ptr(x), _ptr(dy), _ptr(dw), _ptr(db), N, Cin, H, W, Cout, R, 2, R // 2,
                                      prec, _ptr(ws), ws_bytes, _stream()), "conv_small_wgrad")
    return dw, db


class PackedConvWeight:
    """Opaque packed copies of one conv weight (include/b200np.h): `f` forward order, `d` data-gradient
    order, each followed by its tensor-core image for 64x64 layers."""
    __slots__ = ("f", "d", "Cout", "Cin", "R")

    def __init__(self, f, d, Cout, Cin, R):
        self.f, self.d, self.Cout, self.Cin, self.R = f, d, Cout, Cin, R


def pack_conv_weight(w, want_fwd=True, want_dgrad=True):
    """torch [Cout,Cin,R,R] -> PackedConvWeight."""
    _chk(w, "w")
    Cout, Cin, R, _ = w.shape
    n = LIB.b200np_packed_weight_floats(Cout, Cin, R)
    wf = empty((n,), w) if want_fwd else None
    wd = empty((n,), w) if want_dgrad else None
    check(LIB.b200np_pack_conv_weight(_ptr(w), _ptr(wf), _ptr(wd), Cout, Cin, R, _stream()), "pack_conv_weight")
    return PackedConvWeight(wf, wd, Cout, Cin, R)


def conv_fwd(x, pw, bias, stride, act, prec, skip=None, want_bits=False):
    """x NHWC, pw PackedConvWeight; skip = (xs, pws, bias_s, stride_s) fuses a 1x1 projection of xs.
    want_bits: also return the packed gates (y > 0) [N,OH,OW,2] int32 (tensor-core modes, 64 channels) -> (y, bits)."""
    _chk(x, "x"), _chk(pw.f, "wf"), _chk(bias, "bias")
    N, H, W, Cin = x.shape
    assert Cin == pw.Cin
    y = empty((N, H // stride, W // stride, pw.Cout), x)
    xs = wsf = bs = None
    Cs, ss = 0, 1
    if skip is not None:
        xs, pws, bs, ss = skip
        _chk(xs, "xs"), _chk(pws.f, "wsf"), _chk(bs, "bias_s")
        wsf, Cs = pws.f, xs.shape[3]
    bits = None
    if want_bits and prec != lib.PREC_FP32_SIMT and Cin == 64 and pw.Cout == 64:
        bits = torch.empty((N, H // stride, W // stride, 2), device=x.device, dtype=torch.int32)
    check(LIB.b200np_conv_fwd(_ptr(x), _ptr(pw.f), _ptr(bias), _ptr(y), N, H, W, Cin, pw.Cout, pw.R, stride,
                              _ptr(xs), _ptr(wsf), _ptr(bs), Cs, ss, act, prec, _ptr(bits), _stream()), "conv_fwd")
    return (y, bits) if want_bits else y


def conv_dgrad(dy, pw, x_shape, stride, prec, mask_src=None, skip=None, mask_bits=None):
    """dy NHWC [N,H/stride,W/stride,Cout] -> dx [N,H,W,Cin], gated by mask_src > 0;
    skip = (dys, pws, stride_s) adds the gradient through a 1x1 stride_s projection."""
    _chk(dy, "dy"), _chk(pw.d, "wd"), _chk(mask_src, "mask")
    N, H, W, Cin = x_shape
    Cout = dy.shape[3]
    assert Cin == pw.Cin and Cout == pw.Cout
    dx = empty(tuple(x_shape), dy)
    dys = wsd = None
    Cs, ss = 0, 1
    if skip is not None:
        dys, pws, ss = skip
        _chk(dys, "dys"), _chk(pws.d, "wsd")
        wsd, Cs = pws.d, dys.shape[3]
    check(LIB.b200np_conv_dgrad(_ptr(dy), _ptr(pw.d), _ptr(dx), _ptr(mask_src), _ptr(mask_bits), N, H, W, Cin, Cout, pw.R, stride,
                                _ptr(dys), _ptr(wsd), Cs, ss, prec, _stream()), "conv_dgrad")
    return dx


def conv_wgrad(x, dy, R, stride, prec, want_db=True, skip=None):
    """-> (dw [Cout,Cin,R,R], db [Cout] | None, dws [64,64,1,1] | None).  skip = (xs, stride_s) also returns the
    weight gradient of the 1x1 projection of xs that was fused into this conv's output."""
    _chk(x, "x"), _chk(dy, "dy")
    N, H, W, Cin = x.shape
    Cout = dy.shape[3]
    ws_bytes = LIB.b200np_conv_wgrad_workspace(N, H, W, Cin, Cout, R, stride)
    ws = torch.empty(max(ws_bytes // 4, 1), device=x.device, dtype=F32)
    dw = empty((Cout, Cin, R, R), x)
    db = empty((Cout,), x) if want_db else None
    xs = dws = None
    ss = 1
    if skip is not None:
        xs, ss = skip
        _chk(xs, "xs")
        dws = empty((Cout, xs.shape[3], 1, 1), x)
    check(LIB.b200np_conv_wgrad(_ptr(x), _ptr(dy), _ptr(dw), _ptr(db), N, H, W, Cin, Cout, R, stride, _ptr(xs),
                                _ptr(dws), ss, prec, _ptr(ws), ws_bytes, _stream()), "conv_wgrad")
    return dw, db, dws


# ----------------------------------------------------------------------------------------------
# pooling / flatten
# ----------------------------------------------------------------------------------------------
def amp2_flatten_fwd(x, out=None, idx=None):
    _chk(x, "x")
    N, H, W, Cc = x.shape
    out = empty((N, Cc * 4), x) if out is None else out
    idx = empty((N, Cc * 4), x, torch.int32) if idx is None else idx
    check(LIB.b200np_adaptive_maxpool2x2_flatten_fwd(_ptr(x), _ptr(out), _ptr(idx), N, H, W, Cc, _stream()),
          "adaptive_maxpool2x2_flatten_fwd")
    return out, idx


def amp2_flatten_bwd(dout, idx, x_saved, dx):
    _chk(dout, "dout")
    N, H, W, Cc = x_saved.shape
    check(LIB.b200np_adaptive_maxpool2x2_flatten_bwd(_ptr(dout), _ptr(idx), _ptr(x_saved), _ptr(dx), N, H, W, Cc,
                                                     _stream()), "adaptive_maxpool2x2_flatten_bwd")
    return dx


def nhwc_to_nchw_flat(x, out=None):
    _chk(x, "x")
    N, H, W, Cc = x.shape
    out = empty((N, Cc * H * W), x) if out is None else out
    check(LIB.b200np_nhwc_to_nchw_flat(_ptr(x), _ptr(out), N, H, W, Cc, _stream()), "nhwc_to_nchw_flat")
    return out


def nchw_flat_to_nhwc(dout, x_saved, dx, mask=True):
    _chk(dout, "dout")
    N, H, W, Cc = dx.shape
    check(LIB.b200np_nchw_flat_to_nhwc(_ptr(dout), _ptr(x_saved if mask else None), _ptr(dx), N, H, W, Cc,
                                       _stream()), "nchw_flat_to_nhwc")
    return dx


def maxpool2x2_fwd(x):
    _chk(x, "x")
    N, H, W, Cc = x.shape
    y = empty((N, H // 2, W // 2, Cc), x)
    idx = empty((N, H // 2, W // 2, Cc), x, torch.int8)
    check(LIB.b200np_maxpool2x2_fwd(_ptr(x), _ptr(y), _ptr(idx), N, H, W, Cc, _stream()), "maxpool2x2_fwd")
    return y, idx


def maxpool2x2_bwd(dy, idx, x_saved):
    _chk(dy, "dy")
    N, H, W, Cc = x_saved.shape
    dx = empty((N, H, W, Cc), dy)
    check(LIB.b200np_maxpool2x2_bwd(_ptr(dy), _ptr(idx), _ptr(x_saved), _ptr(dx), N, H, W, Cc, _stream()),
          "maxpool2x2_bwd")
    return dx


# ----------------------------------------------------------------------------------------------
# GEMM and friends
# ----------------------------------------------------------------------------------------------
def gemm(A, B, Cmat, M, N, K, a_rs, a_cs, b_rs, b_cs, ldc, bias=None, alpha=1.0, beta=0.0, act=lib.ACT_NONE,
         row_scale=None, addend=None, ld_add=0, prec=lib.PREC_FP32_SIMT, sum_groups=False, conv=None):
    """A, B, Cmat, bias: device pointers (ints) or lists of up to 8 of them (grouped).  sum_groups: the groups
    are K-slices of one product written to Cmat[0].  conv = (operand, H, W, C): operand 1 (A) or 2 (B) is the virtual
    tap-major im2col matrix of the NHWC tensor its pointer addresses (include/b200np.h)."""
    d = GemmDesc()
    As = A if isinstance(A, (list, tuple)) else [A]
    Bs = B if isinstance(B, (list, tuple)) else [B]
    Cs = Cmat if isinstance(Cmat, (list, tuple)) else [Cmat]
    bs = bias if isinstance(bias, (list, tuple)) else [bias] * len(As)
    g = len(As)
    assert len(Bs) == g and len(Cs) == g and len(bs) == g and g <= 8
    for i in range(g):
        d.A[i], d.B[i], d.C[i], d.bias[i] = As[i], Bs[i], Cs[i], bs[i] or 0
    d.groups, d.M, d.N, d.K = g, M, N, K
    d.a_rs, d.a_cs, d.b_rs, d.b_cs, d.ldc = a_rs, a_cs, b_rs, b_cs, ldc
    d.alpha, d.beta, d.act = alpha, beta, act
    d.row_scale = 0 if row_scale is None else row_scale.data_ptr()
    d.addend = 0 if addend is None else addend.data_ptr()
    d.ld_add, d.precision = ld_add, prec
    d.workspace, d.workspace_bytes, d.sum_groups = 0, 0, int(sum_groups)
    d.conv_operand, d.conv_H, d.conv_W, d.conv_C = conv if conv is not None else (0, 0, 0, 0)
    ws_bytes = LIB.b200np_gemm_workspace(C.byref(d))
    if ws_bytes:  # split-K scratch for the GEMMs with too few output tiles to fill the chip
        ws = torch.empty(ws_bytes // 4, device="cuda", dtype=F32)
        d.workspace, d.workspace_bytes = ws.data_ptr(), ws_bytes
    check(LIB.b200np_gemm(C.byref(d), _stream()), "gemm")


def act_bwd(dy, y, act):
    _chk(dy, "dy"), _chk(y, "y")
    dz = torch.empty_like(dy)
    check(LIB.b200np_act_bwd(_ptr(dy), _ptr(y), _ptr(dz), dy.numel(), act, _stream()), "act_bwd")
    return dz


def colsum(x, rows, cols, ld, out=None):
    _chk(x, "x")
    out = empty((cols,), x) if out is None else out
    ws_bytes = LIB.b200np_colsum_workspace(rows, cols)
    ws = torch.empty(max(ws_bytes // 4, 1), device=x.device, dtype=F32)
    check(LIB.b200np_colsum(_ptr(x), _ptr(out), rows, cols, ld, _ptr(ws), ws_bytes, _stream()), "colsum")
    return out


def fill(x, value):
    check(LIB.b200np_fill(_ptr(x), x.numel(), float(value), _stream()), "fill")
    return x


def zeros(shape, like):
    return fill(empty(shape, like), 0.0)


def gather_images_u8(bank, rows, out=None):
    """bank uint8 [n,H,W,C] (CUDA), rows int32 [...] (CUDA) -> fp32 [..., C, H, W] = (255 - bank[rows]) / 255."""
    if not (bank.is_cuda and rows.is_cuda and bank.dtype == torch.uint8 and rows.dtype == torch.int32):
        raise lib.B200NPError("gather_images_u8: needs a CUDA uint8 bank and CUDA int32 row indices")
    if not (bank.is_contiguous() and rows.is_contiguous()):
        raise lib.B200NPError("gather_images_u8: tensors must be contiguous")
    _, H, W, Cc = bank.shape
    if out is None:
        out = torch.empty(tuple(rows.shape) + (Cc, H, W), device=bank.device, dtype=F32)
    check(LIB.b200np_gather_images_u8(_ptr(bank), _ptr(rows), _ptr(out), rows.numel(), H, W, Cc, _stream()),
          "gather_images_u8")
    return out


def _segments(segments):
    """(src, off, n) triples -> the host arrays and count of b200np_multi_copy / b200np_multi_accumulate."""
    k = len(segments)
    srcs = (C.c_void_p * k)(*[None if s is None else s.data_ptr() for s, _, _ in segments])
    offs = (C.c_longlong * k)(*[o for _, o, _ in segments])
    nums = (C.c_longlong * k)(*[n for _, _, n in segments])
    return srcs, offs, nums, k


def multi_copy(dst, segments):
    """dst[off:off+n] = src (zeros for src None) for every (src, off, n) in segments -- one launch per 64."""
    if segments:
        check(LIB.b200np_multi_copy(*_segments(segments), _ptr(dst), _stream()), "multi_copy")
    return dst


def multi_accumulate(dst, segments):
    """dst[off:off+n] += src (src None: left unchanged) for every (src, off, n) in segments -- one launch per 64."""
    if segments:
        check(LIB.b200np_multi_accumulate(*_segments(segments), _ptr(dst), _stream()), "multi_accumulate")
    return dst


def axpy(y, x, a=1.0):
    check(LIB.b200np_axpy(_ptr(y), _ptr(x), y.numel(), float(a), _stream()), "axpy")
    return y


def repeat_rows(x, rep):
    rows, cols = x.shape
    y = empty((rows * rep, cols), x)
    check(LIB.b200np_repeat_rows(_ptr(x), _ptr(y), rows, rep, cols, _stream()), "repeat_rows")
    return y


def repeat_rows_bwd(dy, rep):
    rows, cols = dy.shape[0] // rep, dy.shape[1]
    dx = empty((rows, cols), dy)
    check(LIB.b200np_repeat_rows_bwd(_ptr(dy), _ptr(dx), rows, rep, cols, _stream()), "repeat_rows_bwd")
    return dx


def scale_by_device_scalar(x, s):
    y = torch.empty_like(x)
    check(LIB.b200np_scale_by_device_scalar(_ptr(x), _ptr(s), _ptr(y), x.numel(), _stream()), "scale")
    return y


def reduce(x, op):
    out = empty((1,), x)
    check(LIB.b200np_reduce(_ptr(x), x.numel(), _ptr(out), op, _stream()), "reduce")
    return out


# ----------------------------------------------------------------------------------------------
# aggregation, loss, optimizer
# ----------------------------------------------------------------------------------------------
def ctx_aggregate_fwd(feats, mode):
    _chk(feats, "feats")
    T, nc, D = feats.shape
    out = empty((T, D), feats)
    idx = empty((T, D), feats, torch.int32) if mode == 1 else None
    check(LIB.b200np_ctx_aggregate_fwd(_ptr(feats), _ptr(out), _ptr(idx), T, nc, D, mode, _stream()),
          "ctx_aggregate_fwd")
    return out, idx


def ctx_aggregate_bwd(dout, idx, T, nc, D, mode):
    _chk(dout, "dout")
    df = empty((T, nc, D), dout)
    check(LIB.b200np_ctx_aggregate_bwd(_ptr(dout), _ptr(idx), _ptr(df), T, nc, D, mode, _stream()),
          "ctx_aggregate_bwd")
    return df


def baco_fwd(mu, s):
    _chk(mu, "mu"), _chk(s, "s")
    T, nc, D = mu.shape
    r = empty((T, D), mu)
    check(LIB.b200np_baco_fwd(_ptr(mu), _ptr(s), _ptr(r), T, nc, D, _stream()), "baco_fwd")
    return r


def baco_bwd(dr, mu, s, r):
    _chk(dr, "dr")
    T, nc, D = mu.shape
    dmu, ds = torch.empty_like(mu), torch.empty_like(s)
    check(LIB.b200np_baco_bwd(_ptr(dr), _ptr(mu), _ptr(s), _ptr(r), _ptr(dmu), _ptr(ds), T, nc, D, _stream()), "baco_bwd")
    return dmu, ds


def loss_fwd_bwd(mu, y, kind, want_grad=True):
    _chk(mu, "mu"), _chk(y, "y")
    R = mu.numel() // mu.shape[-1]
    loss = empty((), mu)   # 0-dim, owns its storage (LossFunc hands it out as the loss)
    dmu = torch.empty_like(mu) if want_grad else None
    check(LIB.b200np_loss_fwd_bwd(_ptr(mu), _ptr(y), _ptr(loss), _ptr(dmu), R, mu.shape[-1], y.shape[-1], kind,
                                  _stream()), "loss_fwd_bwd")
    return loss, dmu


def adam_step(p, g, m, v, n, lr, b1, b2, eps, wd, step, grad_scale=1.0):
    check(LIB.b200np_adam_step(_ptr(p), _ptr(g), _ptr(m), _ptr(v), n, lr, b1, b2, eps, wd, step, grad_scale,
                               _stream()), "adam_step")


def adam_step_dev(p, g, m, v, n, lr, b1, b2, eps, wd, step_dev, grad_scale=1.0):
    check(LIB.b200np_adam_step_dev(_ptr(p), _ptr(g), _ptr(m), _ptr(v), n, lr, b1, b2, eps, wd, _ptr(step_dev),
                                   grad_scale, _stream()), "adam_step_dev")


def grad_norm_workspace(n, like):
    """The workspace `grad_norm` takes for an n-float segment, on `like`'s device."""
    return torch.empty(LIB.b200np_grad_norm_workspace(n), device=like.device, dtype=torch.uint8)


def grad_norm(g, n, out, ws, scale=1.0):
    """out[0] = scale * ||g[:n]||_2 (fp64 sums, bitwise repeatable); `ws` from grad_norm_workspace."""
    _chk(g, "g"), _chk(out, "out")
    check(LIB.b200np_grad_norm(_ptr(g), n, scale, _ptr(out), _ptr(ws), ws.numel(), _stream()), "grad_norm")


def adam_step_ctrl(p, g, m, v, n, lr, b1, b2, eps, wd, step_dev, grad_scale=1.0, max_norm=None, norm=None,
                   skipped=None):
    """adam_step_dev with lr a device scalar; clipping to the device scalar `max_norm` and skipping a non-finite step
    (counted in `skipped`) are decided from `norm` = grad_norm(g, scale=grad_scale).  None switches either off."""
    check(LIB.b200np_adam_step_ctrl(_ptr(p), _ptr(g), _ptr(m), _ptr(v), n, _ptr(lr), b1, b2, eps, wd, _ptr(step_dev),
                                    grad_scale, _ptr(max_norm), _ptr(norm), _ptr(skipped), _stream()),
          "adam_step_ctrl")


ADAM_GROUP_FIELDS = ("lr", "weight_decay", "beta1", "beta2", "eps", "decoupled")   # b200np_adam_group, 4 B each


def adam_group_table(groups, device):
    """The device table b200np_adam_step_groups reads: a float32 [len(groups), 6] tensor, one b200np_adam_group per
    row, from dicts with torch.optim.Adam's keys.  The `decoupled` column holds an int32 (write it through
    `.view(torch.int32)`)."""
    rows = torch.tensor([[g["lr"], g["weight_decay"], *g["betas"], g["eps"], 0.0] for g in groups], dtype=F32)
    rows.view(torch.int32)[:, 5] = torch.tensor([int(bool(g["decoupled_weight_decay"])) for g in groups],
                                                dtype=torch.int32)
    return rows.to(device)


def adam_step_groups(p, g, m, v, n, groups, run_begin, run_group, step_dev, grad_scale=1.0, max_norm=None, norm=None,
                     skipped=None):
    """adam_step_ctrl with every hyperparameter read per parameter group from the device table `groups`
    (adam_group_table).  Run r of the segment, [run_begin[r], run_begin[r + 1]) (int64, multiples of 4, 0 .. n), is
    updated with group run_group[r] (int32; -1: frozen, left untouched)."""
    for t, name in ((p, "p"), (g, "g"), (m, "m"), (v, "v"), (groups, "groups"), (run_group, "run_group")):
        _chk(t, name)
    if run_begin.dtype != torch.int64 or not run_begin.is_cuda or run_group.dtype != torch.int32 \
            or run_begin.numel() != run_group.numel() + 1 or groups.shape[1:] != (len(ADAM_GROUP_FIELDS),):
        raise lib.B200NPError("adam_step_groups: malformed group or run table")
    check(LIB.b200np_adam_step_groups(_ptr(p), _ptr(g), _ptr(m), _ptr(v), n, _ptr(groups), groups.shape[0],
                                      _ptr(run_begin), _ptr(run_group), run_group.numel(), _ptr(step_dev),
                                      grad_scale, _ptr(max_norm), _ptr(norm), _ptr(skipped), _stream()),
          "adam_step_groups")


# ----------------------------------------------------------------------------------------------
# MMAML conv nets (SURVEY.md 8f-3): im2col / col2im for 3x3 stride-2 convs, batch-stat norm + scale/shift + ReLU
# ----------------------------------------------------------------------------------------------
def im2col3x3s2(x):
    """x NHWC [N,H,W,C] -> col [N*(H/2)*(W/2), C*9] with k = ci*9 + r*3 + s (torch's weight flattening)."""
    _chk(x, "x")
    N, H, W, Cc = x.shape
    col = empty((N * (H // 2) * (W // 2), Cc * 9), x)
    check(LIB.b200np_im2col3x3s2(_ptr(x), _ptr(col), N, H, W, Cc, _stream()), "im2col3x3s2")
    return col


def col2im3x3s2(dcol, x_shape, mask=None):
    _chk(dcol, "dcol"), _chk(mask, "mask")
    N, H, W, Cc = x_shape
    dx = empty(tuple(x_shape), dcol)
    check(LIB.b200np_col2im3x3s2(_ptr(dcol), _ptr(mask), _ptr(dx), N, H, W, Cc, _stream()), "col2im3x3s2")
    return dx


def im2col_small(x, R, pad, ld=None):
    """x NCHW [N, Cin, H, W] -> col [N*(H/2)*(W/2), ld] for an R x R stride-2 convolution (k = ci*R*R + r*R + s, the
    flattening of torch's weight); ld defaults to Cin*R*R rounded up to a multiple of 4."""
    _chk(x, "x")
    N, Cin, H, W = x.shape
    ld = (Cin * R * R + 3) // 4 * 4 if ld is None else ld
    col = empty((N * (H // 2) * (W // 2), ld), x)
    check(LIB.b200np_im2col_small(_ptr(x), _ptr(col), N, Cin, H, W, R, pad, ld, _stream()), "im2col_small")
    return col


def conv_weight_tapmajor(w, to_tapmajor=True):
    """[Cout, Cin, 3, 3] -> [Cout, 9 * Cin] with k = tap * Cin + ci, or back (same shapes reversed)."""
    _chk(w, "w")
    if to_tapmajor:
        Cout, Cin = w.shape[0], w.shape[1]
        out = empty((Cout, 9 * Cin), w)
    else:
        Cout, Cin = w.shape[0], w.shape[1] // 9
        out = empty((Cout, Cin, 3, 3), w)
    check(LIB.b200np_conv_weight_tapmajor(_ptr(w), _ptr(out), Cout, Cin, int(to_tapmajor), _stream()), "conv_weight_tapmajor")
    return out


def col2im3x3s2_tapmajor(dcol, x_shape, mask=None):
    _chk(dcol, "dcol"), _chk(mask, "mask")
    N, H, W, Cc = x_shape
    dx = empty(tuple(x_shape), dcol)
    check(LIB.b200np_col2im3x3s2_tapmajor(_ptr(dcol), _ptr(mask), _ptr(dx), N, H, W, Cc, _stream()), "col2im3x3s2_tapmajor")
    return dx


def bn_act_fwd(x, scale, shift, plus_one, relu=True, eps=1e-5, run_mean=None, run_var=None, momentum=0.1):
    """x [..., C] (rows = everything but the last dim) -> (y, mean [2C], rstd [C]); `mean` holds the batch mean as a
    (hi, lo) pair of floats per channel (hi = mean[:C]), see include/b200np.h."""
    _chk(x, "x"), _chk(scale, "scale"), _chk(shift, "shift")
    Cc = x.shape[-1]
    rows = x.numel() // Cc
    y = torch.empty_like(x)
    mean, rstd = empty((2 * Cc,), x), empty((Cc,), x)
    ws_bytes = LIB.b200np_bn_workspace(rows, Cc)
    ws = torch.empty(max(ws_bytes // 4, 1), device=x.device, dtype=F32)
    check(LIB.b200np_bn_act_fwd(_ptr(x), _ptr(scale), _ptr(shift), float(plus_one), float(eps), _ptr(y), _ptr(mean),
                                _ptr(rstd), _ptr(run_mean), _ptr(run_var), float(momentum), rows, Cc, int(relu),
                                _ptr(ws), ws_bytes, _stream()), "bn_act_fwd")
    return y, mean, rstd


def bn_act_bwd(dy, y, x, mean, rstd, scale, plus_one, relu=True):
    """-> (dx, dscale [C], dshift [C])."""
    _chk(dy, "dy")
    Cc = x.shape[-1]
    rows = x.numel() // Cc
    dx = torch.empty_like(x)
    dscale, dshift = empty((Cc,), x), empty((Cc,), x)
    ws_bytes = LIB.b200np_bn_workspace(rows, Cc)
    ws = torch.empty(max(ws_bytes // 4, 1), device=x.device, dtype=F32)
    check(LIB.b200np_bn_act_bwd(_ptr(dy), _ptr(y), _ptr(x), _ptr(mean), _ptr(rstd), _ptr(scale), float(plus_one), _ptr(dx),
                                _ptr(dscale), _ptr(dshift), rows, Cc, int(relu), _ptr(ws), ws_bytes, _stream()),
          "bn_act_bwd")
    return dx, dscale, dshift


def bn_act_bwd2(dy, y, x, mean, rstd, scale, plus_one, relu, vx, vs, vt, want_x=True, want_dy=True, want_scale=True):
    """Second order: gradients of <vx, dx> + <vs, dscale> + <vt, dshift> (the outputs of bn_act_bwd) with respect to
    x, dy and scale -> (gx, gdy, gscale); vx / vs / vt may be None (zero cotangent)."""
    _chk(dy, "dy")
    Cc = x.shape[-1]
    rows = x.numel() // Cc
    gx = torch.empty_like(x) if want_x else None
    gdy = torch.empty_like(x) if want_dy else None
    gscale = empty((Cc,), x) if want_scale else None
    ws_bytes = LIB.b200np_bn_workspace2(rows, Cc)
    ws = torch.empty(max(ws_bytes // 4, 1), device=x.device, dtype=F32)
    check(LIB.b200np_bn_act_bwd2(_ptr(dy), _ptr(y), _ptr(x), _ptr(mean), _ptr(rstd), _ptr(scale), float(plus_one), _ptr(vx),
                                 _ptr(vs), _ptr(vt), _ptr(gx), _ptr(gdy), _ptr(gscale), rows, Cc, int(relu), _ptr(ws),
                                 ws_bytes, _stream()), "bn_act_bwd2")
    return gx, gdy, gscale


def mul3(a, b=None, c=None, alpha=1.0):
    """alpha * a * b * c elementwise (b, c optional)."""
    _chk(a, "a")
    out = torch.empty_like(a)
    check(LIB.b200np_mul3(_ptr(a), _ptr(b), _ptr(c), float(alpha), _ptr(out), a.numel(), _stream()), "mul3")
    return out


# ----------------------------------------------------------------------------------------------
# Bayes-by-backprop weight sampling + KL (SURVEY.md 8f-4)
# ----------------------------------------------------------------------------------------------
def bbb_sample_kl_fwd(mu, rho, eps, prior_mu, prior_sigma):
    """-> (w = mu + eps * softplus(rho), sigma, kl [1])."""
    _chk(mu, "mu"), _chk(rho, "rho"), _chk(eps, "eps")
    n = mu.numel()
    w, sigma = torch.empty_like(mu), torch.empty_like(mu)
    part = empty((LIB.b200np_bbb_kl_blocks(n),), mu)
    check(LIB.b200np_bbb_sample_kl_fwd(_ptr(mu), _ptr(rho), _ptr(eps), float(prior_mu), float(prior_sigma), _ptr(w),
                                       _ptr(sigma), _ptr(part), n, _stream()), "bbb_sample_kl_fwd")
    return w, sigma, reduce(part, 1)


def bbb_sample_kl_bwd(dw, dkl, mu, rho, eps, sigma, prior_mu, prior_sigma):
    n = mu.numel()
    dmu, drho = torch.empty_like(mu), torch.empty_like(mu)
    check(LIB.b200np_bbb_sample_kl_bwd(_ptr(dw), _ptr(dkl), _ptr(mu), _ptr(rho), _ptr(eps), _ptr(sigma), float(prior_mu),
                                       float(prior_sigma), _ptr(dmu), _ptr(drho), n, _stream()), "bbb_sample_kl_bwd")
    return dmu, drho
