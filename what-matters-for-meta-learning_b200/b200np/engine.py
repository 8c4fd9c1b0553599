"""Forward / backward of the neural-process families on libb200np kernels.

Each segment of the model (CNN trunk, dense layer, head projections, aggregation, FAVOR+
attention, loss) is one ``torch.autograd.Function`` whose forward AND backward are explicit
sequences of C-ABI kernel launches on torch's current stream; torch autograd only stitches the
segments together (views / reshapes -- no ATen compute kernels on the path).  Nothing here
falls back to PyTorch ops: without the CUDA library or a CUDA tensor the calls raise.

Reference call sites mirrored: networks/models.py:92-117,156-192 (CNN), networks/ResNet.py:58-74
(BasicBlock), networks/ANPDistractor.py:78-135, networks/CNPDistractor.py:77-124,
networks/CNPShapeNet1D.py:95-143, networks/ANPShapeNet1D.py:93-161,
networks/fast_attention.py:74-99,151-156.
"""
import os

import torch
from torch.autograd import Function

from . import dist, ops
from .lib import ACT_NONE, ACT_RELU, ACT_TANH, PREC_FP32_SIMT, PREC_TF32, PREC_TF32X3

_PREC_NAMES = {"fp32": PREC_FP32_SIMT, "tf32x3": PREC_TF32X3, "tf32": PREC_TF32}
PRECISION = _PREC_NAMES[os.environ.get("B200NP_PRECISION", "tf32x3")]


def set_precision(name):
    """'tf32x3' (fp32-grade 3-pass split on tcgen05, default), 'tf32' (single pass, what cuDNN's
    default does for the reference on Ampere+), or 'fp32' (CUDA-core kernels, validation)."""
    global PRECISION
    PRECISION = _PREC_NAMES[name]


def _p(t, off=0):
    return t.data_ptr() + 4 * off


# NVTX ranges around the segments of the step (B200NP_NVTX=1): names show up in Nsight Systems / ncu --nvtx timelines
# next to the kernels of each segment.  Off by default: a push/pop pair per segment costs ~1 us of host time.
NVTX = os.environ.get("B200NP_NVTX", "0") == "1"


class nvtx_range:
    def __init__(self, name):
        self.name = name

    def __enter__(self):
        if NVTX:
            torch.cuda.nvtx.range_push(self.name)

    def __exit__(self, *exc):
        if NVTX:
            torch.cuda.nvtx.range_pop()
        return False


# The decoder's CNN (networks/models.py:160-180) depends on the target images only, so it runs on a second stream
# beside the encoder CNN / attention / MLP chain of the main stream and joins where `fc_mu` consumes it.  Autograd runs
# each backward node on its forward stream, so the two trunks' backward passes overlap the same way; inside a captured
# step the fork/join becomes two branches of the CUDA graph.  The big persistent conv kernels still take turns on the
# SMs -- what overlaps are the latency-bound kernels of one branch (small maps, partial reductions, dense layers,
# FAVOR+) with the other branch, and every kernel's tail.  B200NP_OVERLAP=0 keeps everything on one stream.
#
# Level 2 (default): inside a trunk's backward pass the weight gradients are off the critical path (only the
# data-gradient chain feeds the next layer), so they are issued on a companion stream of the stream the backward node
# runs on and join before the node returns.
OVERLAP = int(os.environ.get("B200NP_OVERLAP", "2"))
_SIDE = {}


# Stream priorities (CUDA clamps them to the device's range; captured kernel nodes inherit them): the stream that
# carries the encoder CNN -> attention -> loss chain should win SMs over the decoder branch, and a trunk's data-gradient
# chain over its weight gradients, so the companions only fill what the critical chain leaves idle.  The caller's own
# stream has the default (lowest) priority in eager mode; `optim.GraphedStep` captures on a stream of MAIN_PRIORITY.
MAIN_PRIORITY, DECODER_PRIORITY, WGRAD_PRIORITY = -2, -1, 0
USE_PRIORITIES = os.environ.get("B200NP_PRIO", "1") != "0"


# Called at the start of every CNN trunk's backward with the data pointer of the trunk's first parameter.  By then every
# gradient that does not belong to a trunk is complete (the trunks are the leaves of the backward pass), so a data-parallel
# optimizer starts their all-reduce here and lets it run beside the trunk's backward (b200np/optim.py: FusedAdam).
PRE_TRUNK_BACKWARD_HOOKS = []


def _pre_trunk_backward(ptr):
    for hook in list(PRE_TRUNK_BACKWARD_HOOKS):
        hook(ptr)


def _side_stream(key, priority=0):
    """One lazily created companion stream per key (the role and the handle of the stream it accompanies)."""
    s = _SIDE.get(key)
    if s is None:
        s = _SIDE[key] = torch.cuda.Stream(priority=priority if USE_PRIORITIES else 0)
    return s


# ================================================================================================
# CNN trunk: stem 5x5 s2 + 4 residual stages + pooling, several image sources in one pass
# ================================================================================================
class TrunkFn(Function):
    @staticmethod
    def forward(ctx, img_agg, prec, n_src, *tensors):
        with nvtx_range("b200np.trunk.forward"):
            return TrunkFn._forward(ctx, img_agg, prec, n_src, *tensors)

    @staticmethod
    def _forward(ctx, img_agg, prec, n_src, *tensors):
        imgs, params = tensors[:n_src], tensors[n_src:]
        assert len(params) == 26
        if img_agg not in ("max", "baco", "reshape"):
            # 'mean' yields 64 features and breaks the 256-wide Linear in the reference too
            raise NotImplementedError(f"img_agg={img_agg!r} is unusable in the reference (SURVEY.md 8a/a1)")
        c1w, c1b = params[0], params[1]
        Ns = [im.shape[0] for im in imgs]
        N = sum(Ns)
        _, H, W = imgs[0].shape[1:]
        x0 = ops.empty((N, H // 2, W // 2, 64), imgs[0])
        # 1-bit ReLU gates of the stem output: the stride-2 data gradient of layer1 ends in this tensor and would
        # otherwise re-read all of it (1 MB per image) just for the sign
        bits0 = None
        if ops.relu_bits_supported(imgs[0].shape[1], c1w.shape[2], c1w.shape[0], prec):
            bits0 = torch.empty((N, H // 2, W // 2, 2), device=x0.device, dtype=torch.int32)
        off = 0
        # Stems the tcgen05 stem kernel does not cover (3-channel tasks: 5x5 over RGB, K = 75) in the tensor-core modes:
        # im2col of the thin NCHW input + the tcgen05 GEMM with a fused bias + ReLU epilogue, and dW = dY^T col in the
        # backward -- the CUDA-core direct convolution and its weight gradient were 22 % of the ShapeNet3D step
        stem_cols = [] if (prec != PREC_FP32_SIMT and bits0 is None) else None
        for im, n in zip(imgs, Ns):
            if stem_cols is not None:
                R, K = c1w.shape[2], c1w.shape[1] * c1w.shape[2] * c1w.shape[3]
                col = ops.im2col_small(im.contiguous(), R, R // 2)
                ops.gemm(_p(col), _p(c1w), _p(x0[off:off + n]), col.shape[0], c1w.shape[0], K, col.shape[1], 1, 1, K,
                         c1w.shape[0], bias=_p(c1b), act=ACT_RELU, prec=prec)
                stem_cols.append(col)
            else:
                ops.conv_small_fwd(im, c1w, c1b, out=x0[off:off + n], relu=True, prec=prec,
                                   relu_bits=None if bits0 is None else bits0[off:off + n])
            off += n
        ctx.stem_cols = stem_cols
        x, acts, packs, bits, bits_x = x0, [], [], [], bits0
        for l in range(4):
            w1, b1, w2, b2, wsk, bsk = params[2 + 6 * l: 8 + 6 * l]
            p1, p2, ps = ops.pack_conv_weight(w1), ops.pack_conv_weight(w2), ops.pack_conv_weight(wsk)
            # the forward epilogues also emit the ReLU gates as 1 bit per element (None in fp32 mode): the data
            # gradients read those instead of the activations
            h, bits_h = ops.conv_fwd(x, p1, b1, 2, ACT_RELU, prec, want_bits=True)
            y, bits_y = ops.conv_fwd(h, p2, b2, 1, ACT_RELU, prec, skip=(x, ps, bsk, 2), want_bits=True)
            acts.append((x, h, y))
            bits.append((bits_x, bits_h))
            packs.append((p1, p2, ps))
            x, bits_x = y, bits_y
        outs, idxs, off = [], [], 0
        for n in Ns:
            xs = x[off:off + n]
            if img_agg == "reshape":
                outs.append(ops.nhwc_to_nchw_flat(xs))
                idxs.append(None)
            else:
                o, i = ops.amp2_flatten_fwd(xs)
                outs.append(o)
                idxs.append(i)
            off += n
        ctx.img_agg, ctx.prec, ctx.Ns = img_agg, prec, Ns
        ctx.first_param_ptr = c1w.data_ptr()
        ctx.imgs, ctx.acts, ctx.packs, ctx.idxs, ctx.bits = imgs, acts, packs, idxs, bits
        ctx.c1w_shape = tuple(c1w.shape)
        ctx.pool_idx = idxs  # exposed for parity tests (bit-exact argmax)
        return tuple(outs)

    @staticmethod
    def backward(ctx, *douts):
        with nvtx_range("b200np.trunk.backward"):
            return TrunkFn._backward(ctx, *douts)

    @staticmethod
    def _backward(ctx, *douts):
        prec, Ns = ctx.prec, ctx.Ns
        _pre_trunk_backward(ctx.first_param_ptr)
        y_last = ctx.acts[3][2]
        dy = torch.empty_like(y_last)
        off = 0
        for n, do, idx in zip(Ns, douts, ctx.idxs):
            do = do.contiguous()
            if ctx.img_agg == "reshape":
                ops.nchw_flat_to_nhwc(do, y_last[off:off + n], dy[off:off + n])
            else:
                ops.amp2_flatten_bwd(do, idx, y_last[off:off + n], dy[off:off + n])
            off += n
        grads = [None] * 26
        cur = torch.cuda.current_stream()
        wst = _side_stream(("wgrad", cur.cuda_stream), WGRAD_PRIORITY) if OVERLAP >= 2 else None
        if wst is None:
            wst = cur
            fork = join = lambda: None
        else:
            fork, join = (lambda: wst.wait_stream(cur)), (lambda: cur.wait_stream(wst))
        keep = []   # tensors the companion stream reads stay referenced until it has joined (allocator reuse is per stream)
        for l in (3, 2, 1, 0):
            x, h, _ = ctx.acts[l]
            p1, p2, ps = ctx.packs[l]
            bits_x, bits_h = ctx.bits[l]
            fork()
            with torch.cuda.stream(wst):
                if prec == PREC_FP32_SIMT:
                    dw2, db2, _ = ops.conv_wgrad(h, dy, 3, 1, prec)
                    dws, _, _ = ops.conv_wgrad(x, dy, 1, 2, prec, want_db=False)
                else:  # the skip projection's weight gradient rides along as a 10th tap of conv2's
                    dw2, db2, dws = ops.conv_wgrad(h, dy, 3, 1, prec, skip=(x, 2))
                dbs = db2.clone()
            dh = ops.conv_dgrad(dy, p2, h.shape, 1, prec, mask_src=h, mask_bits=bits_h)
            fork()
            with torch.cuda.stream(wst):
                dw1, db1, _ = ops.conv_wgrad(x, dh, 3, 2, prec)
            dx = ops.conv_dgrad(dh, p1, x.shape, 2, prec, mask_src=x, skip=(dy, ps, 2), mask_bits=bits_x)
            grads[2 + 6 * l: 8 + 6 * l] = [dw1, db1, dw2, db2, dws, dbs]
            keep += [dy, dh]
            dy = dx
        fork()
        off, dw_acc, db_acc = 0, None, None
        with torch.cuda.stream(wst):
            for si, (im, n) in enumerate(zip(ctx.imgs, Ns)):
                if ctx.stem_cols is not None:
                    col, dyv = ctx.stem_cols[si], dy[off:off + n]
                    Co, K, M = ctx.c1w_shape[0], col.shape[1], col.shape[0]
                    Kw = ctx.c1w_shape[1] * ctx.c1w_shape[2] * ctx.c1w_shape[3]
                    dw = ops.empty(ctx.c1w_shape, dyv)
                    ops.gemm(_p(dyv), _p(col), _p(dw), Co, Kw, M, 1, Co, K, 1, Kw, prec=prec)      # dW = dY^T col
                    db = ops.colsum(dyv, M, Co, Co)
                else:
                    dw, db = ops.conv_small_wgrad(im, dy[off:off + n], ctx.c1w_shape, prec)
                if dw_acc is None:
                    dw_acc, db_acc = dw, db
                else:
                    ops.axpy(dw_acc, dw)
                    ops.axpy(db_acc, db)
                off += n
        join()
        del keep
        grads[0], grads[1] = dw_acc, db_acc
        return (None, None, None) + (None,) * len(Ns) + tuple(grads)


class EncoderW0Fn(Function):
    """encoder_w0 up to (and including) nn.Flatten: conv 1->32 s2, conv 32->48 s2, maxpool 2x2,
    conv 48->64 s2, NCHW flatten (networks/CNPShapeNet1D.py:46-55).  The trailing Linear 4096->dim_w
    is a LinearFn."""

    @staticmethod
    def forward(ctx, prec, n_src, *tensors):
        imgs = tensors[:n_src]
        w0, b0, w2, b2, w5, b5 = tensors[n_src:]
        Ns = [im.shape[0] for im in imgs]
        N = sum(Ns)
        _, H, W = imgs[0].shape[1:]
        x1 = ops.empty((N, H // 2, W // 2, w0.shape[0]), imgs[0])
        # the sources (context / target images) as ONE batch: one launch of the first conv and of its weight gradient
        # instead of one per source (20 MB copied once against two half-filled launches each way)
        img_all = imgs[0].contiguous() if n_src == 1 else torch.cat([im.reshape(im.shape[0], -1) for im in imgs]).view(
            N, *imgs[0].shape[1:])
        ops.conv_small_fwd(img_all, w0, b0, out=x1, relu=True, prec=prec)
        if prec == PREC_FP32_SIMT:
            wd2, wd5 = ops.pack_conv_weight(w2), ops.pack_conv_weight(w5)
            x2 = ops.conv_fwd(x1, wd2, b2, 2, ACT_RELU, prec)
            x3, pidx = ops.maxpool2x2_fwd(x2)
            x4 = ops.conv_fwd(x3, wd5, b5, 2, ACT_RELU, prec)
        else:
            # 32 -> 48 and 48 -> 64 channels do not fill the 64 x 64 tap-convolution tiles: the tcgen05 GEMM with a VIRTUAL
            # im2col operand (b200np_gemm_desc.conv_operand: k = tap*C + ci, gathered as 16-byte words while the operand
            # is staged) and a fused bias + ReLU epilogue -- no column matrix is written or read (it was 354 MB for the
            # 32 -> 48 layer of 300 images, written once and read twice per step)
            wd2 = wd5 = None
            w2, w5 = ops.conv_weight_tapmajor(w2), ops.conv_weight_tapmajor(w5)      # [Cout, 9*Cin], tap-major
            M2, K2 = N * (H // 4) * (W // 4), w2.shape[1]
            x2 = ops.empty((N, H // 4, W // 4, w2.shape[0]), imgs[0])
            ops.gemm(_p(x1), _p(w2), _p(x2), M2, w2.shape[0], K2, K2, 1, 1, K2, w2.shape[0], bias=_p(b2), act=ACT_RELU,
                     prec=prec, conv=(1, H // 2, W // 2, x1.shape[-1]))
            x3, pidx = ops.maxpool2x2_fwd(x2)
            M5, K5 = N * (H // 16) * (W // 16), w5.shape[1]
            x4 = ops.empty((N, H // 16, W // 16, w5.shape[0]), imgs[0])
            ops.gemm(_p(x3), _p(w5), _p(x4), M5, w5.shape[0], K5, K5, 1, 1, K5, w5.shape[0], bias=_p(b5), act=ACT_RELU,
                     prec=prec, conv=(1, H // 8, W // 8, x3.shape[-1]))
        outs, off = [], 0
        for n in Ns:
            outs.append(ops.nhwc_to_nchw_flat(x4[off:off + n]))
            off += n
        ctx.prec, ctx.Ns, ctx.imgs = prec, Ns, img_all
        ctx.first_param_ptr = w0.data_ptr()
        ctx.saved = (x1, x2, x3, x4, pidx, wd2, wd5, tuple(w0.shape), w2, w5)
        return tuple(outs)

    @staticmethod
    def backward(ctx, *douts):
        prec, Ns = ctx.prec, ctx.Ns
        _pre_trunk_backward(ctx.first_param_ptr)
        x1, x2, x3, x4, pidx, wd2, wd5, w0_shape, w2, w5 = ctx.saved
        d4 = torch.empty_like(x4)
        off = 0
        for n, do in zip(Ns, douts):
            ops.nchw_flat_to_nhwc(do.contiguous(), x4[off:off + n], d4[off:off + n])
            off += n
        if wd2 is not None:
            dw5, db5, _ = ops.conv_wgrad(x3, d4, 3, 2, prec)
            d3 = ops.conv_dgrad(d4, wd5, x3.shape, 2, prec, mask_src=None)
            d2 = ops.maxpool2x2_bwd(d3, pidx, x2)
            dw2, db2, _ = ops.conv_wgrad(x1, d2, 3, 2, prec)
            d1 = ops.conv_dgrad(d2, wd2, x1.shape, 2, prec, mask_src=x1)
        else:
            def conv_bwd(x_in, wt, dy, mask):     # wt: tap-major [Cout, 9*Cin]; x_in NHWC, the conv's input
                Co, K = wt.shape
                M = dy.numel() // Co
                _, Hi, Wi, Ci = x_in.shape
                dwt = ops.empty((Co, K), wt)
                ops.gemm(_p(dy), _p(x_in), _p(dwt), Co, K, M, 1, Co, K, 1, K, prec=prec, conv=(2, Hi, Wi, Ci))   # dW = dY^T col(x)
                db = ops.colsum(dy, M, Co, Co)
                dcol = ops.empty((M, K), dy)
                ops.gemm(_p(dy), _p(wt), _p(dcol), M, K, Co, Co, 1, K, 1, K, prec=prec)                            # dcol = dY W
                return ops.conv_weight_tapmajor(dwt, to_tapmajor=False), db, ops.col2im3x3s2_tapmajor(dcol, x_in.shape, mask=mask)
            dw5, db5, d3 = conv_bwd(x3, w5, d4, None)
            d2 = ops.maxpool2x2_bwd(d3, pidx, x2)
            dw2, db2, d1 = conv_bwd(x1, w2, d2, x1)
        dw0, db0 = ops.conv_small_wgrad(ctx.imgs, d1, w0_shape, prec)
        return (None, None) + (None,) * len(Ns) + (dw0, db0, dw2, db2, dw5, db5)


# ================================================================================================
# dense layers
# ================================================================================================
class LinearFn(Function):
    """y = act([x, x2] @ w^T + b): nn.Linear (+ torch.cat of two inputs, + ReLU/Tanh) in one kernel."""

    @staticmethod
    def forward(ctx, act, prec, x_in, x2, w, b):
        x = x_in.contiguous()
        K1 = x.shape[-1]
        rows = x.numel() // K1
        N, Kt = w.shape
        y = ops.empty(tuple(x.shape[:-1]) + (N,), x)
        if x2 is None:
            assert Kt == K1
            ops.gemm(_p(x), _p(w), _p(y), rows, N, K1, K1, 1, 1, Kt, N, bias=_p(b), act=act, prec=prec)
        else:
            x2 = x2.contiguous()
            K2 = x2.shape[-1]
            assert Kt == K1 + K2 and x2.numel() // K2 == rows
            ops.gemm(_p(x), _p(w), _p(y), rows, N, K1, K1, 1, 1, Kt, N, prec=prec)
            ops.gemm(_p(x2), _p(w, K1), _p(y), rows, N, K2, K2, 1, 1, Kt, N, bias=_p(b), beta=1.0, act=act,
                     prec=prec)
        ctx.act, ctx.prec, ctx.rows = act, prec, rows
        ctx.x_is_input = x is x_in
        ctx.save_for_backward(x, x2, w, y)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, x2, w, y = ctx.saved_tensors
        act, prec, rows = ctx.act, ctx.prec, ctx.rows
        if torch.is_grad_enabled():      # create_graph=True (second-order MAML): differentiable backward ops
            from . import second_order
            if x2 is not None or not ctx.x_is_input:
                raise NotImplementedError("second-order gradients of a dense layer need one contiguous input")
            dx, dw, db = second_order.linear_backward(act, prec, x, w, y, dy, ctx.needs_input_grad[2])
            return None, None, dx, None, dw, db
        dy = dy.contiguous()
        dz = ops.act_bwd(dy, y, act) if act != ACT_NONE else dy
        N, Kt = w.shape
        K1 = x.shape[-1]
        dx = dx2 = None
        if ctx.needs_input_grad[2]:
            dx = torch.empty_like(x)
            ops.gemm(_p(dz), _p(w), _p(dx), rows, K1, N, N, 1, Kt, 1, K1, prec=prec)
        dw = ops.empty((N, Kt), w)
        ops.gemm(_p(dz), _p(x), _p(dw), N, K1, rows, 1, N, K1, 1, Kt, prec=prec)
        if x2 is not None:
            K2 = x2.shape[-1]
            if ctx.needs_input_grad[3]:
                dx2 = torch.empty_like(x2)
                ops.gemm(_p(dz), _p(w, K1), _p(dx2), rows, K2, N, N, 1, Kt, 1, K2, prec=prec)
            ops.gemm(_p(dz), _p(x2), _p(dw, K1), N, K2, rows, 1, N, K2, 1, Kt, prec=prec)
        db = ops.colsum(dz, rows, N, N)
        return None, None, dx, dx2, dw, db


class HeadsLinearFn(Function):
    """Eight per-head nn.Linear(K -> d) applied to the same rows (networks/ANPDistractor.py:83-96)
    as one grouped GEMM; output [rows, H*d] with head h in columns [h*d, (h+1)*d)."""

    @staticmethod
    def forward(ctx, prec, x, *wb):
        H = len(wb) // 2
        ws, bs = wb[:H], wb[H:]
        x = x.contiguous()
        K = x.shape[-1]
        rows = x.numel() // K
        d = ws[0].shape[0]
        y = ops.empty((rows, H * d), x)
        ops.gemm([_p(x)] * H, [_p(w) for w in ws], [_p(y, h * d) for h in range(H)], rows, d, K, K, 1, 1, K, H * d,
                 bias=[_p(b) for b in bs], prec=prec)
        ctx.prec, ctx.rows, ctx.H, ctx.d = prec, rows, H, d
        ctx.save_for_backward(x, *ws)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, *ws = ctx.saved_tensors
        prec, rows, H, d = ctx.prec, ctx.rows, ctx.H, ctx.d
        K = x.shape[-1]
        dy = dy.contiguous()
        dw = ops.empty((H, d, K), x)
        ops.gemm([_p(dy, h * d) for h in range(H)], [_p(x)] * H, [_p(dw, h * d * K) for h in range(H)], d, K, rows,
                 1, H * d, K, 1, K, prec=prec)
        db = ops.colsum(dy, rows, H * d, H * d)
        dx = None
        if ctx.needs_input_grad[1]:
            dx = torch.empty_like(x)  # dX = sum_h dY_h W_h: the heads are K-slices of one product
            ops.gemm([_p(dy, h * d) for h in range(H)], [_p(w) for w in ws], [_p(dx)] * H, rows, K, d, H * d, 1, K, 1, K,
                     prec=prec, sum_groups=True)
        return (None, dx) + tuple(dw[h] for h in range(H)) + tuple(db[h * d:(h + 1) * d] for h in range(H))


class AggregateFn(Function):
    """mean / max over the context dimension (networks/CNPDistractor.py:96-101)."""

    @staticmethod
    def forward(ctx, mode, feats):
        feats = feats.contiguous()
        out, idx = ops.ctx_aggregate_fwd(feats, mode)
        ctx.mode, ctx.shape, ctx.idx = mode, feats.shape, idx
        return out

    @staticmethod
    def backward(ctx, dout):
        T, nc, D = ctx.shape
        if torch.is_grad_enabled():      # create_graph=True
            from . import second_order
            if ctx.mode != 0:
                raise NotImplementedError("second-order gradients are implemented for the mean aggregation only")
            return None, second_order.MeanBwdP.apply(dout, nc)
        return None, ops.ctx_aggregate_bwd(dout.contiguous(), ctx.idx, T, nc, D, ctx.mode)


class BacoFn(Function):
    """Bayesian context aggregation (networks/CNPDistractor.py:60-75,104-110): mu, s [T,nc,D] -> r [T,D]."""

    @staticmethod
    def forward(ctx, mu, s):
        mu, s = mu.contiguous(), s.contiguous()
        r = ops.baco_fwd(mu, s)
        ctx.save_for_backward(mu, s, r)
        return r

    @staticmethod
    def backward(ctx, dr):
        mu, s, r = ctx.saved_tensors
        return ops.baco_bwd(dr.contiguous(), mu, s, r)


class RepeatFn(Function):
    """x[:, None, :].repeat(1, rep, 1) (networks/CNPDistractor.py:99)."""

    @staticmethod
    def forward(ctx, rep, x):
        ctx.rep = rep
        return ops.repeat_rows(x.contiguous(), rep)

    @staticmethod
    def backward(ctx, dy):
        return None, ops.repeat_rows_bwd(dy.contiguous(), ctx.rep)


# ================================================================================================
# FAVOR+ attention (networks/fast_attention.py:74-99,151-156,187-205)
# ================================================================================================
class FavorAttentionFn(Function):
    """q [T*nt, H*d], k, v [T*nc, H*d] (head-major columns) -> out [T*nt, d*H] (index e*H + h)."""

    @staticmethod
    def forward(ctx, prec, T, H, nt, nc, xq, xk, v, proj):
        with nvtx_range("b200np.favor.forward"):
            return FavorAttentionFn._forward(ctx, prec, T, H, nt, nc, xq, xk, v, proj)

    @staticmethod
    def _forward(ctx, prec, T, H, nt, nc, xq, xk, v, proj):
        if prec == PREC_TF32:
            prec = PREC_TF32X3  # the feature pre-activations go through exp(): always fp32-grade (SURVEY.md section 7)
        xq, xk, v = xq.contiguous(), xk.contiguous(), v.contiguous()
        M, d = proj.shape
        ldu = (M + 3) // 4 * 4
        Rq, Rk = T * nt * H, T * nc * H
        c = float(d) ** -0.25
        U = ops.empty((Rq, ldu), xq)
        W = ops.empty((Rk, ldu), xq)
        ops.gemm(_p(xq), _p(proj), _p(U), Rq, M, d, d, 1, 1, d, ldu, alpha=c, prec=prec)
        ops.gemm(_p(xk), _p(proj), _p(W), Rk, M, d, d, 1, 1, d, ldu, alpha=c, prec=prec)
        sq, mq, amq = ops.empty((Rq,), xq), ops.empty((Rq,), xq), ops.empty((Rq,), xq, torch.int32)
        tk, mk = ops.empty((Rk,), xq), ops.empty((Rk,), xq)
        ops.check(ops.LIB.b200np_favor_rowstats(ops._ptr(xq), ops._ptr(U), ops._ptr(sq), ops._ptr(mq), ops._ptr(amq),
                                                Rq, d, M, ldu, ops._stream()), "favor_rowstats(q)")
        ops.check(ops.LIB.b200np_favor_rowstats(ops._ptr(xk), ops._ptr(W), ops._ptr(tk), ops._ptr(mk), ops._ptr(None),
                                                Rk, d, M, ldu, ops._stream()), "favor_rowstats(k)")
        g = ops.reduce(mk, 0)
        dist.all_reduce_max(g)  # the key stabiliser is a max over the WHOLE meta-batch (fast_attention.py:97)
        ties = ops.zeros((1,), xq)
        out = ops.empty((T * nt, d * H), xq)
        A = ops.empty((T * H * nt * nc,), xq)
        Dn = ops.empty((T * H * nt,), xq)
        ops.check(ops.LIB.b200np_favor_attn_fwd(*(ops._ptr(t) for t in (U, W, sq, mq, tk, g, v, out, A, Dn, ties)),
                                                T, H, nt, nc, d, M, ldu, ops._stream()), "favor_attn_fwd")
        ctx.dims = (prec, T, H, nt, nc, d, M, ldu)
        ctx.save_for_backward(xq, xk, v, proj, U, W, sq, mq, amq, tk, g, out, A, Dn, ties)
        return out

    @staticmethod
    def backward(ctx, d_out):
        xq, xk, v, proj, U, W, sq, mq, amq, tk, g, out, A, Dn, ties = ctx.saved_tensors
        prec, T, H, nt, nc, d, M, ldu = ctx.dims
        Rq, Rk = T * nt * H, T * nc * H
        c = float(d) ** -0.25
        d_out = d_out.contiguous()
        dU, dW = ops.empty((Rq, ldu), xq), ops.empty((Rk, ldu), xq)
        dv = torch.empty_like(v)
        ds, dt = ops.empty((Rq,), xq), ops.empty((Rk,), xq)
        dg_part = ops.empty((T * H,), xq)
        ops.check(ops.LIB.b200np_favor_attn_bwd(
            *(ops._ptr(t) for t in (d_out, U, W, sq, mq, amq, tk, g, v, out, A, Dn, dU, dW, dv, ds, dt, dg_part)),
            T, H, nt, nc, d, M, ldu, ops._stream()), "favor_attn_bwd")
        dg = ops.reduce(dg_part, 1)
        tie_total = ties
        if dist.world_size() > 1:
            # d loss / d g and the tie count both sum over every rank's keys: ONE 8-byte all-reduce, not two
            pair = ops.empty((2,), xq)
            ops.multi_copy(pair, [(dg, 0, 1), (ties, 1, 1)])
            dist.all_reduce_sum(pair)
            dg, tie_total = pair[0:1], pair[1:2]
        ops.check(ops.LIB.b200np_favor_key_fixup(ops._ptr(dW), ops._ptr(W), ops._ptr(g), ops._ptr(dg),
                                                 ops._ptr(tie_total), Rk, M, ldu, ops._stream()), "favor_key_fixup")
        dxq, dxk = torch.empty_like(xq), torch.empty_like(xk)
        ops.gemm(_p(dU), _p(proj), _p(dxq), Rq, d, M, ldu, 1, d, 1, d, alpha=c, row_scale=ds, addend=xq, ld_add=d,
                 prec=prec)
        ops.gemm(_p(dW), _p(proj), _p(dxk), Rk, d, M, ldu, 1, d, 1, d, alpha=c, row_scale=dt, addend=xk, ld_add=d,
                 prec=prec)
        return None, None, None, None, None, dxq, dxk, dv, None


# ================================================================================================
# model families
# ================================================================================================
def _lin(act, x, x2, layer):
    return LinearFn.apply(act, PRECISION, x, x2, layer.weight, layer.bias)


def _trunk_params(holder):
    ps = [holder.conv1.weight, holder.conv1.bias]
    for st in holder.resnet.stages():
        ps += [st.conv1.weight, st.conv1.bias, st.conv2.weight, st.conv2.bias,
               st.downsample[0].weight, st.downsample[0].bias]
    return ps


def _heads(x, heads):
    return HeadsLinearFn.apply(PRECISION, x, *[m.linear.weight for m in heads], *[m.linear.bias for m in heads])


def _attention(m, T, nt, nc, k_in, v_in, q_in):
    """_multihead_attention (networks/ANPDistractor.py:78-101)."""
    H = m.n_heads
    k = _heads(k_in, m._W_k)
    v = _heads(v_in, m._W_v)
    q = _heads(q_in, m._W_q)
    att = FavorAttentionFn.apply(PRECISION, T, H, nt, nc, q, k, v, m.attn.projection_matrix)
    return _lin(ACT_NONE, att, None, m._W.linear)


def _check_inputs(m, ctx_x, ctx_y, tgt_x):
    for t, name in ((ctx_x, "context images"), (ctx_y, "context labels"), (tgt_x, "target images")):
        if not (torch.is_tensor(t) and t.is_cuda and t.dtype == torch.float32):
            raise RuntimeError(f"{name}: expected a float32 CUDA tensor (the B200 path has no CPU fallback)")
    if tgt_x.shape[0] != m.task_num:
        raise RuntimeError(f"batch has {tgt_x.shape[0]} tasks but config.tasks_per_batch={m.task_num} "
                           "(same constraint as networks/models.py:115)")


def _forward_resnet_family(m, ctx_x, ctx_y, tgt_x):
    T, nc, nt = m.task_num, ctx_x.shape[1], tgt_x.shape[1]
    C, H, W = m.img_channels, m.img_size[0], m.img_size[1]
    tgt_imgs = tgt_x.reshape(T * nt, C, H, W).contiguous()
    dec_params = _trunk_params(m.decoder)
    side = None
    if OVERLAP >= 1 and nc:
        main = torch.cuda.current_stream()
        side = _side_stream(("decoder", main.cuda_stream), DECODER_PRIORITY)
        side.wait_stream(main)
        with torch.cuda.stream(side):
            (x_dec,) = TrunkFn.apply(m.img_agg, PRECISION, 1, tgt_imgs, *dec_params)
    if nc:
        ctx_imgs = ctx_x.reshape(T * nc, C, H, W).contiguous()
        lab = ctx_y.reshape(T * nc, -1).contiguous()
        if hasattr(m, "transform_y"):
            lab = _lin(ACT_NONE, lab, None, m.transform_y)
        enc = _trunk_params(m.img_encoder)
        if m.attention:
            x_ctx, x_tgt = TrunkFn.apply(m.img_agg, PRECISION, 2, ctx_imgs, tgt_imgs, *enc)
        else:
            if m.agg_mode not in ("mean", "max", "baco"):
                raise TypeError("agg_mode is not applicable for CNP, choose from ['mean', 'max', 'baco']")
            (x_ctx,) = TrunkFn.apply(m.img_agg, PRECISION, 1, ctx_imgs, *enc)
        cf = _lin(ACT_RELU, x_ctx, lab, m.task_encoder[0])
        cf = _lin(ACT_RELU, cf, None, m.task_encoder[2])
        cf = _lin(ACT_RELU, cf, None, m.task_encoder[4])
        if m.attention:
            rep = _attention(m, T, nt, nc, x_ctx, cf, x_tgt)
            sample = _lin(ACT_NONE, rep, None, m.mu)
        else:
            if m.agg_mode == "baco":   # CNPDistractor.py:104-110
                lm = _lin(ACT_NONE, cf, None, m.latent_mu)
                ls = _lin(ACT_NONE, cf, None, m.latent_var)
                r = BacoFn.apply(lm.view(T, nc, -1), ls.view(T, nc, -1))
            else:
                r = AggregateFn.apply(0 if m.agg_mode == "mean" else 1, cf.view(T, nc, -1))
            sample = RepeatFn.apply(nt, _lin(ACT_NONE, r, None, m.mu))
    else:
        sample = ops.zeros((T * nt, 256), tgt_imgs)
    if side is not None:
        main.wait_stream(side)
    else:
        (x_dec,) = TrunkFn.apply(m.img_agg, PRECISION, 1, tgt_imgs, *dec_params)
    fc = m.decoder.fc_mu
    h = _lin(ACT_RELU, x_dec, sample, fc[0])
    h = _lin(ACT_RELU, h, None, fc[2])
    out = _lin(ACT_NONE, h, None, fc[4])
    return out.view(T, nt, -1)


def _forward_shapenet1d_family(m, ctx_x, ctx_y, tgt_x):
    T, nc, nt = m.task_num, ctx_x.shape[1], tgt_x.shape[1]
    C, H, W = m.img_channels, m.img_size[0], m.img_size[1]
    e = m.encoder_w0
    conv_params = [e[0].weight, e[0].bias, e[2].weight, e[2].bias, e[5].weight, e[5].bias]
    tgt_imgs = tgt_x.reshape(T * nt, C, H, W).contiguous()
    if nc:
        ctx_imgs = ctx_x.reshape(T * nc, C, H, W).contiguous()
        f_ctx, f_tgt = EncoderW0Fn.apply(PRECISION, 2, ctx_imgs, tgt_imgs, *conv_params)
        x_ctx = _lin(ACT_NONE, f_ctx, None, e[8])
        x_qry = _lin(ACT_NONE, f_tgt, None, e[8])
        lab = _lin(ACT_NONE, ctx_y.reshape(T * nc, -1).contiguous(), None, m.transform_y)
        L = m.encoder_r.layers
        rs = _lin(ACT_RELU, x_ctx, lab, L[0])
        rs = _lin(ACT_RELU, rs, None, L[2])
        rs = _lin(ACT_NONE, rs, None, L[4])
        if m.attention:
            if m.agg_mode != "attention":
                raise TypeError("agg_mode is not applicable for CNP, choose from ['attention']")
            r = _attention(m, T, nt, nc, x_ctx, rs, x_qry)
            z = _lin(ACT_NONE, r, None, m.r_to_z)
        else:
            if m.agg_mode == "baco":
                # CNPShapeNet1D.py:74-76 builds rs_to_mu / rs_to_var as Linear(256, 256) but feeds them dim_r-wide
                # features (100 in every shipped config): the reference itself fails on this path
                raise NotImplementedError("agg_mode='baco' is shape-inconsistent in the reference's ShapeNet1D CNP "
                                          "(SURVEY.md 8a/a8)")
            if m.agg_mode not in ("mean", "max"):
                raise TypeError("agg_mode is not applicable for CNP, choose from ['mean', 'max', 'baco']")
            r = AggregateFn.apply(0 if m.agg_mode == "mean" else 1, rs.view(T, nc, -1))
            z = RepeatFn.apply(nt, _lin(ACT_NONE, r, None, m.r_to_z))
    else:
        (f_tgt,) = EncoderW0Fn.apply(PRECISION, 1, tgt_imgs, *conv_params)
        x_qry = _lin(ACT_NONE, f_tgt, None, e[8])
        z = ops.zeros((T * nt, m.dim_z), tgt_imgs)
    D = m.decoder0
    h = _lin(ACT_RELU, x_qry, z, D[0])
    h = _lin(ACT_RELU, h, None, D[2])
    out = _lin(ACT_TANH, h, None, D[4])
    return out.view(T, nt, -1)


def forward(model, ctx_x, ctx_y, tgt_x):
    _check_inputs(model, ctx_x, ctx_y, tgt_x)
    with nvtx_range(f"b200np.forward[{type(model).__name__}]"):
        if model.family == "resnet":
            return _forward_resnet_family(model, ctx_x, ctx_y, tgt_x)
        return _forward_shapenet1d_family(model, ctx_x, ctx_y, tgt_x)
