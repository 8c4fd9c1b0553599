"""Which kernel computes each conv, stem and GEMM form, and whether it computes it right.

Every dispatcher of the library treats B200NP_E_UNSUPPORTED from a kernel as "try the next one" (halo -> gather ->
CUDA cores for the convolutions, tcgen05 -> CUDA cores for the GEMM), so a kernel that started refusing every shape
would still give correct numbers, only slower.  Each case here therefore pins the kernels that ran (torch.profiler
names) besides checking the result against fp64 torch on the GPU.  The cases call the C ABI directly on guarded
buffers, one allocation [guard | payload | guard] each:

  - input guards hold a NaN pattern, so a read past the end of an input shows up as NaN in the output;
  - output and workspace guards must be bit-identical after the call (no write past the end);
  - outputs and workspaces are poisoned before each of two runs, first with NaN, then with a finite value: an
    element that is never written, or a workspace element read before it is written, makes the two runs differ;
    the two runs must also agree bit for bit because the library promises deterministic reductions;
  - payloads start either 256-B aligned or 16-B but not 32-B aligned (the ABI promises only 16 B).

Bars: 2e-5 relative L2 for fp32 and tf32x3, 3e-3 for single-pass tf32, 4e-5 for weight gradients over >= 1e5 pixels;
integer results bit-exact.
"""
import collections
import ctypes as C
import glob
import importlib
import os
import re

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

PRECS = {"fp32": 0, "tf32x3": 1, "tf32": 2}
TC_PRECS = ("tf32x3", "tf32")
BAR = {"fp32": 2e-5, "tf32x3": 2e-5, "tf32": 3e-3}
BIG_WGRAD_PIXELS = 100_000

GUARD = 1024                                   # bytes of guard on each side of a payload
FLOAT_GUARD = 0x7FA5A5A5                       # a NaN bit pattern
INT_GUARD = 0xA5A5A5A5 - (1 << 32)             # 0xA5 bytes
POISON = {torch.float32: (0x7FC0BAD0, float("-3e38")), torch.int32: (0x5A5A5A5A, -0x5A5A5A5B)}
OFFSETS = {"a256": 0, "a16": 16}               # payload offset past a 512-B aligned guard


# ------------------------------------------------------------------------------------------------
# harness
# ------------------------------------------------------------------------------------------------
def _lib():
    from b200np import lib
    return lib


def normalize(name):
    """'void (anonymous namespace)::k<true, 9, 6>((anonymous namespace)::A, B)' -> 'k<true, 9, 6>'."""
    s = name.replace("(anonymous namespace)::", "").replace("<unnamed>::", "")
    if s.startswith("void "):
        s = s[5:]
    depth = 0
    for i, ch in enumerate(s):
        if ch == "<":
            depth += 1
        elif ch == ">":
            depth -= 1
        elif ch == "(" and depth == 0:
            s = s[:i]
            break
    head, sep, tail = s.partition("<")
    return head.rsplit("::", 1)[-1] + sep + tail


def launched(fn):
    """Runs fn under torch.profiler and returns the normalized names of the CUDA kernels it launched."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [normalize(ev.name) for ev in prof.events() if ev.device_type == torch.autograd.DeviceType.CUDA]


class Guarded:
    """One allocation [guard | payload | guard].  role: 'in' (payload given), 'out' / 'ws' (poisoned before each run),
    'inout' (read and written: restored to its initial value before each run)."""

    def __init__(self, role, shape, dtype=torch.float32, init=None, offset=0):
        self.role, self.shape, self.dtype = role, tuple(shape), dtype
        numel = 1
        for s in self.shape:
            numel *= s
        self.nbytes = numel * 4
        self.off = GUARD + offset
        total = self.off + self.nbytes + GUARD
        self.raw = torch.empty(total // 4, dtype=torch.int32, device="cuda")
        self.raw.fill_(FLOAT_GUARD if dtype == torch.float32 else INT_GUARD)
        self.bytes = self.raw.view(torch.uint8)
        self.payload = self.bytes[self.off:self.off + self.nbytes].view(dtype).view(self.shape)
        if init is not None:
            self.payload.copy_(init.reshape(self.shape))
        self.initial = self.payload.clone()

    @property
    def ptr(self):
        return self.payload.data_ptr()

    def cptr(self):
        return C.c_void_p(self.ptr)

    def guards(self):
        return self.bytes[:self.off], self.bytes[self.off + self.nbytes:]

    def bits(self):
        return self.payload.view(torch.int32)


def rel_l2(got, ref):
    got, ref = got.double(), ref.double()
    return float((got - ref).norm() / ref.norm().clamp_min(1e-300))


class Spec:
    """What one case runs: call() issues the C-ABI call(s); bufs are every Guarded buffer it touches; refs maps an
    output name to (fp64 reference, bar); exact maps an output name to a function of the outputs giving the
    bit-exact expectation."""

    def __init__(self, call, bufs, refs, exact=None):
        self.call, self.bufs, self.refs, self.exact = call, bufs, refs, exact or {}


def run_case(spec, expect=None):
    """Runs spec twice and checks guards, full writes, determinism, inputs, routes and parity.  Raises
    AssertionError naming what went wrong; returns {'kernels': [...], 'rel': {output: rel-L2}}."""
    bufs = spec.bufs
    outs = {n: b for n, b in bufs.items() if b.role in ("out", "inout")}
    results, kernels = [], None
    for run in range(2):
        for b in bufs.values():
            if b.role in ("out", "ws"):
                poison = POISON[b.dtype][run]
                (b.bits() if isinstance(poison, int) else b.payload).fill_(poison)
            elif b.role == "inout":
                b.payload.copy_(b.initial)
        torch.cuda.synchronize()
        snap = {n: b.raw.clone() for n, b in bufs.items()}
        if run == 0:
            kernels = launched(spec.call)
        else:
            spec.call()
            torch.cuda.synchronize()
        for n, b in bufs.items():
            sb = snap[n].view(torch.uint8)
            lo, hi = b.guards()
            if not (torch.equal(lo, sb[:b.off]) and torch.equal(hi, sb[b.off + b.nbytes:])):
                raise AssertionError(f"guard of '{n}' overwritten (run {run})")
            if b.role == "in" and not torch.equal(b.bits(), b.initial.view(torch.int32)):
                raise AssertionError(f"input '{n}' modified (run {run})")
        results.append({n: b.payload.clone() for n, b in outs.items()})
    for n, b in outs.items():
        r0, r1 = results[0][n], results[1][n]
        if b.dtype == torch.float32:
            for run, r in enumerate((r0, r1)):
                if bool(torch.isnan(r).any()):
                    raise AssertionError(f"output '{n}' has NaN in run {run}: not fully written, or it read a "
                                         "guard or an unwritten workspace element")
        if not torch.equal(r0.view(torch.int32), r1.view(torch.int32)):
            raise AssertionError(f"output '{n}' differs between runs with different poison: not fully written, or "
                                 "not deterministic")
    got = results[1]
    if expect is not None:
        seen, want = collections.Counter(kernels), collections.Counter(expect)
        if seen != want:
            raise AssertionError(f"kernels: expected {dict(want)}, launched {dict(seen)}")
    rels = {}
    for n, (ref, bar) in spec.refs.items():
        rels[n] = rel_l2(got[n], ref)
    for n, fn in spec.exact.items():
        if not torch.equal(got[n], fn(got)):
            raise AssertionError(f"output '{n}' is not bit-exact")
    bad = {n: (rels[n], bar) for n, (_, bar) in spec.refs.items() if not rels[n] < bar}
    if bad:
        raise AssertionError(f"rel-L2 over the bar: {bad}")
    return {"kernels": kernels, "rel": rels}


# ------------------------------------------------------------------------------------------------
# inputs and references
# ------------------------------------------------------------------------------------------------
def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def rnd(shape, seed, scale=1.0, sign=False):
    """Zero-mean normal data, or with sign=True uniform [0, 1) -- what a layer sees after a ReLU."""
    g = _gen(seed)
    t = torch.rand(shape, generator=g, device="cuda") if sign else torch.randn(shape, generator=g, device="cuda")
    return t * scale


def nchw(t):
    return t.permute(0, 3, 1, 2).double()


def nhwc(t):
    return t.permute(0, 2, 3, 1).contiguous()


def pack_bits(act):
    """[..., 64] -> int32 [..., 2]: bit j of word h = (act[..., 32h + j] > 0) (include/b200np.h)."""
    g = (act > 0).to(torch.int64).reshape(*act.shape[:-1], 2, 32)
    w = (g << torch.arange(32, device=g.device, dtype=torch.int64)).sum(-1)
    return torch.where(w >= 2 ** 31, w - 2 ** 32, w).to(torch.int32).contiguous()


def packed(w):
    from b200np import ops
    return ops.pack_conv_weight(w.contiguous())


# ------------------------------------------------------------------------------------------------
# case builders: one per entry point
# ------------------------------------------------------------------------------------------------
def conv_fwd_spec(prec, N, H, W, stride, cin=64, cout=64, skip=False, bits=False, sign=False, off=0, seed=1):
    lib = _lib()
    P = PRECS[prec]
    OH, OW = H // stride, W // stride
    x = rnd((N, H, W, cin), seed, sign=sign)
    w = rnd((cout, cin, 3, 3), seed + 1, 0.05, sign)
    b = rnd((cout,), seed + 2, 0.1)
    pw = packed(w)
    bufs = {"x": Guarded("in", x.shape, init=x, offset=off), "wf": Guarded("in", pw.f.shape, init=pw.f, offset=off),
            "b": Guarded("in", b.shape, init=b, offset=off), "y": Guarded("out", (N, OH, OW, cout), offset=off)}
    ref = F.conv2d(nchw(x), w.double(), b.double(), stride=stride, padding=1)
    if skip:
        xs = rnd((N, 2 * OH, 2 * OW, cin), seed + 3, sign=sign)
        wsk = rnd((cout, cin, 1, 1), seed + 4, 0.1, sign)
        bs = rnd((cout,), seed + 5, 0.1)
        bufs["xs"] = Guarded("in", xs.shape, init=xs, offset=off)
        bufs["wsf"] = Guarded("in", packed(wsk).f.shape, init=packed(wsk).f, offset=off)
        bufs["bs"] = Guarded("in", bs.shape, init=bs, offset=off)
        ref = ref + F.conv2d(nchw(xs), wsk.double(), bs.double(), stride=2)
    if bits:
        bufs["bits"] = Guarded("out", (N, OH, OW, 2), torch.int32, offset=off)
    ref = nhwc(F.relu(ref))
    B = bufs.get

    def call():
        lib.check(lib.LIB.b200np_conv_fwd(
            B("x").cptr(), B("wf").cptr(), B("b").cptr(), B("y").cptr(), N, H, W, cin, cout, 3, stride,
            B("xs").cptr() if skip else None, B("wsf").cptr() if skip else None, B("bs").cptr() if skip else None,
            cin if skip else 0, 2, lib.ACT_RELU, P, B("bits").cptr() if bits else None, None), "conv_fwd")
    exact = {"bits": lambda o: pack_bits(o["y"])} if bits else {}
    return Spec(call, bufs, {"y": (ref, BAR[prec])}, exact)


def conv_dgrad_spec(prec, N, H, W, stride, cin=64, cout=64, skip=False, mask=None, off=0, seed=11):
    """dx [N,H,W,cin] from dy [N,H/stride,W/stride,cout]; mask: None, 'src' (float activation) or 'bits'."""
    lib = _lib()
    P = PRECS[prec]
    OH, OW = H // stride, W // stride
    dy = rnd((N, OH, OW, cout), seed)
    w = rnd((cout, cin, 3, 3), seed + 1, 0.05)
    pw = packed(w)
    bufs = {"dy": Guarded("in", dy.shape, init=dy, offset=off), "wd": Guarded("in", pw.d.shape, init=pw.d, offset=off),
            "dx": Guarded("out", (N, H, W, cin), offset=off)}
    ref = torch.nn.grad.conv2d_input((N, cin, H, W), w.double(), nchw(dy), stride=stride, padding=1)
    if skip:
        dys = rnd((N, OH, OW, cout), seed + 2)
        wsk = rnd((cout, cin, 1, 1), seed + 3, 0.1)
        bufs["dys"] = Guarded("in", dys.shape, init=dys, offset=off)
        bufs["wsd"] = Guarded("in", packed(wsk).d.shape, init=packed(wsk).d, offset=off)
        ref = ref + torch.nn.grad.conv2d_input((N, cin, H, W), wsk.double(), nchw(dys), stride=2)
    if mask is not None:
        act = rnd((N, H, W, cin), seed + 4)
        ref = ref * (nchw(act) > 0)
        if mask == "src":
            bufs["mask"] = Guarded("in", act.shape, init=act, offset=off)
        else:
            bufs["mbits"] = Guarded("in", (N, H, W, 2), torch.int32, init=pack_bits(act), offset=off)
    B = bufs.get

    def call():
        lib.check(lib.LIB.b200np_conv_dgrad(
            B("dy").cptr(), B("wd").cptr(), B("dx").cptr(), B("mask").cptr() if mask == "src" else None,
            B("mbits").cptr() if mask == "bits" else None, N, H, W, cin, cout, 3, stride,
            B("dys").cptr() if skip else None, B("wsd").cptr() if skip else None, cout if skip else 0,
            stride, P, None), "conv_dgrad")
    return Spec(call, bufs, {"dx": (nhwc(ref), BAR[prec])})


def conv_wgrad_spec(prec, N, H, W, stride, cin=64, cout=64, R=3, skip=False, sign=False, off=0, seed=21):
    lib = _lib()
    P = PRECS[prec]
    OH, OW = H // stride, W // stride
    x = rnd((N, H, W, cin), seed, sign=sign)
    dy = rnd((N, OH, OW, cout), seed + 1, sign=sign)
    wsb = lib.LIB.b200np_conv_wgrad_workspace(N, H, W, cin, cout, R, stride)
    bufs = {"x": Guarded("in", x.shape, init=x, offset=off), "dy": Guarded("in", dy.shape, init=dy, offset=off),
            "dw": Guarded("out", (cout, cin, R, R), offset=off), "db": Guarded("out", (cout,), offset=off),
            "ws": Guarded("ws", (wsb // 4,), offset=off)}
    pixels = N * OH * OW
    bar = max(BAR[prec], 4e-5) if pixels >= BIG_WGRAD_PIXELS else BAR[prec]
    refs = {"dw": (torch.nn.grad.conv2d_weight(nchw(x), (cout, cin, R, R), nchw(dy), stride=stride, padding=R // 2), bar),
            "db": (dy.double().sum((0, 1, 2)), bar)}
    if skip:
        xs = rnd((N, 2 * OH, 2 * OW, cin), seed + 2, sign=sign)
        bufs["xs"] = Guarded("in", xs.shape, init=xs, offset=off)
        bufs["dws"] = Guarded("out", (cout, cin, 1, 1), offset=off)
        refs["dws"] = (torch.nn.grad.conv2d_weight(nchw(xs), (cout, cin, 1, 1), nchw(dy), stride=2), bar)
    B = bufs.get

    def call():
        lib.check(lib.LIB.b200np_conv_wgrad(
            B("x").cptr(), B("dy").cptr(), B("dw").cptr(), B("db").cptr(), N, H, W, cin, cout, R, stride,
            B("xs").cptr() if skip else None, B("dws").cptr() if skip else None, 2, P, B("ws").cptr(), wsb, None),
            "conv_wgrad")
    return Spec(call, bufs, refs)


def stem_spec(prec, N, cin, H, W, R, cout, bits=False, off=0, seed=31):
    """conv_small_fwd (stride 2, pad R/2, ReLU) and its weight gradient, in one case."""
    lib = _lib()
    P = PRECS[prec]
    OH, OW = H // 2, W // 2
    x = rnd((N, cin, H, W), seed)
    w = rnd((cout, cin, R, R), seed + 1, 0.2)
    b = rnd((cout,), seed + 2)
    dy = rnd((N, OH, OW, cout), seed + 3)
    wsb = lib.LIB.b200np_conv_small_wgrad_workspace(N, cin, H, W, cout, R, 2, R // 2, P)
    bufs = {"x": Guarded("in", x.shape, init=x, offset=off), "w": Guarded("in", w.shape, init=w, offset=off),
            "b": Guarded("in", b.shape, init=b, offset=off), "dy": Guarded("in", dy.shape, init=dy, offset=off),
            "y": Guarded("out", (N, OH, OW, cout), offset=off), "dw": Guarded("out", w.shape, offset=off),
            "db": Guarded("out", (cout,), offset=off), "ws": Guarded("ws", (max(wsb // 4, 1),), offset=off)}
    if bits:
        bufs["bits"] = Guarded("out", (N, OH, OW, 2), torch.int32, offset=off)
    y_ref = nhwc(F.relu(F.conv2d(x.double(), w.double(), b.double(), stride=2, padding=R // 2)))
    dw_ref = torch.nn.grad.conv2d_weight(x.double(), w.shape, nchw(dy), stride=2, padding=R // 2)
    tc = prec != "fp32" and (cin, R, cout) == (1, 5, 64)
    bar = BAR[prec] if tc else BAR["fp32"]
    B = bufs.get

    def call():
        lib.check(lib.LIB.b200np_conv_small_fwd(B("x").cptr(), B("w").cptr(), B("b").cptr(), B("y").cptr(), N, cin, H, W,
                                                cout, R, 2, R // 2, 1, P, B("bits").cptr() if bits else None, None),
                  "conv_small_fwd")
        lib.check(lib.LIB.b200np_conv_small_wgrad(B("x").cptr(), B("dy").cptr(), B("dw").cptr(), B("db").cptr(), N, cin,
                                                  H, W, cout, R, 2, R // 2, P, B("ws").cptr(), wsb, None),
                  "conv_small_wgrad")
    exact = {"bits": lambda o: pack_bits(o["y"])} if bits else {}
    return Spec(call, bufs, {"y": (y_ref, bar), "dw": (dw_ref, bar), "db": (dy.double().sum((0, 1, 2)), bar)}, exact)


def gemm_spec(prec, M, N, K, role="fwd", pad_a=0, bias=False, act=0, alpha=1.0, beta=0.0, row_scale=False,
              groups=1, conv=None, sign=False, off=0, seed=41):
    """C[M,N] = act(alpha * A @ B + bias + beta * C + row_scale * addend).  role: 'fwd' (A k-contiguous, B = W [N,K]),
    'dgrad' (A k-contiguous, B [K,N] n-contiguous), 'wgrad' (A m-contiguous, B [K,N] n-contiguous).  groups > 1:
    the groups are K-slices of one product (sum_groups).  conv = (operand, H, W, C, images): implicit 3x3 stride-2
    convolution with operand 1 (forward: A) or 2 (weight gradient: B) virtual."""
    lib = _lib()
    P = PRECS[prec]
    bufs, refs = {}, {}
    d = lib.GemmDesc()
    if conv is None:
        A = rnd((M, K), seed, sign=sign)
        Bm = rnd((K, N), seed + 1, 0.1, sign)
        if role == "fwd":
            lda, ldb = K + pad_a, K
            a_store, b_store = F.pad(A, (0, pad_a)), Bm.t()
            d.a_rs, d.a_cs, d.b_rs, d.b_cs = lda, 1, 1, ldb
        elif role == "dgrad":
            lda, ldb = K + pad_a, N
            a_store, b_store = F.pad(A, (0, pad_a)), Bm
            d.a_rs, d.a_cs, d.b_rs, d.b_cs = lda, 1, ldb, 1
        else:
            lda, ldb = M + pad_a, N
            a_store, b_store = F.pad(A.t(), (0, pad_a)), Bm
            d.a_rs, d.a_cs, d.b_rs, d.b_cs = 1, lda, ldb, 1
        bufs["A"] = Guarded("in", a_store.shape, init=a_store.contiguous(), offset=off)
        bufs["B"] = Guarded("in", b_store.shape, init=b_store.contiguous(), offset=off)
        prod = A.double() @ Bm.double()
        Kg = K // groups
        for g in range(groups):     # group g = K-slice g (role dgrad: A columns, B rows)
            d.A[g] = bufs["A"].ptr + 4 * g * Kg * (d.a_cs if role == "wgrad" else 1)
            d.B[g] = bufs["B"].ptr + 4 * g * Kg * (d.b_rs if role != "fwd" else 1)
    else:
        operand, cH, cW, cC, imgs = conv
        x = rnd((imgs, cH, cW, cC), seed, sign=sign)
        bufs["x"] = Guarded("in", x.shape, init=x, offset=off)
        if operand == 1:     # y[M, N=Cout] = im2col(x) @ W^T, W tap-major [Cout, 9C]
            w = rnd((N, cC, 3, 3), seed + 1, 0.1, sign)
            wt = w.permute(0, 2, 3, 1).reshape(N, 9 * cC).contiguous()
            bufs["B"] = Guarded("in", wt.shape, init=wt, offset=off)
            d.A[0], d.B[0] = bufs["x"].ptr, bufs["B"].ptr
            d.a_rs, d.a_cs, d.b_rs, d.b_cs = K, 1, 1, K
            prod = nhwc(F.conv2d(nchw(x), w.double(), stride=2, padding=1)).reshape(M, N)
        else:                # dW[M=Cout, N=9C] = dY^T @ im2col(x)
            dy = rnd((imgs, cH // 2, cW // 2, M), seed + 1, sign=sign)
            bufs["A"] = Guarded("in", dy.shape, init=dy, offset=off)
            d.A[0], d.B[0] = bufs["A"].ptr, bufs["x"].ptr
            d.a_rs, d.a_cs, d.b_rs, d.b_cs = 1, M, N, 1
            dw = torch.nn.grad.conv2d_weight(nchw(x), (M, cC, 3, 3), nchw(dy), stride=2, padding=1)
            prod = dw.permute(0, 2, 3, 1).reshape(M, N)
        d.conv_operand, d.conv_H, d.conv_W, d.conv_C = operand, cH, cW, cC
    c0 = rnd((M, N), seed + 2)
    bufs["C"] = Guarded("inout" if beta else "out", (M, N), init=c0, offset=off)
    ref = alpha * prod
    if bias:
        bv = rnd((N,), seed + 3)
        bufs["bias"] = Guarded("in", bv.shape, init=bv, offset=off)
        ref = ref + bv.double()
        d.bias[0] = bufs["bias"].ptr
    if beta:
        ref = ref + beta * c0.double()
    if row_scale:
        rs, add = rnd((M,), seed + 4), rnd((M, N), seed + 5)
        bufs["rs"] = Guarded("in", rs.shape, init=rs, offset=off)
        bufs["add"] = Guarded("in", add.shape, init=add, offset=off)
        ref = ref + rs.double()[:, None] * add.double()
        d.row_scale, d.addend, d.ld_add = bufs["rs"].ptr, bufs["add"].ptr, N
    ref = {0: ref, 1: F.relu(ref), 2: torch.tanh(ref)}[act]
    for g in range(groups):
        d.C[g] = bufs["C"].ptr
    d.groups, d.sum_groups = groups, int(groups > 1)
    d.M, d.N, d.K = M, N, (K // groups if groups > 1 else K)
    d.ldc, d.alpha, d.beta, d.act, d.precision = N, alpha, beta, act, P
    wsb = lib.LIB.b200np_gemm_workspace(C.byref(d))
    if wsb:
        bufs["ws"] = Guarded("ws", (wsb // 4,), offset=off)
        d.workspace, d.workspace_bytes = bufs["ws"].ptr, wsb
    big = conv is not None and conv[0] == 2 and K >= BIG_WGRAD_PIXELS

    def call():
        lib.check(lib.LIB.b200np_gemm(C.byref(d), None), "gemm")
    return Spec(call, bufs, {"C": (ref, max(BAR[prec], 4e-5) if big else BAR[prec])})


def ctx_agg_spec(prec, T, nc, D, mode, off=0, seed=51):
    lib = _lib()
    f = F.relu(rnd((T, nc, D), seed))
    bufs = {"f": Guarded("in", f.shape, init=f, offset=off), "out": Guarded("out", (T, D), offset=off)}
    if mode == 1:
        bufs["idx"] = Guarded("out", (T, D), torch.int32, offset=off)
    ref, ridx = (f.double().mean(1), None) if mode == 0 else f.max(1)
    exact = {} if mode == 0 else {"idx": lambda o: ridx.to(torch.int32), "out": lambda o: ref}
    B = bufs.get

    def call():
        lib.check(lib.LIB.b200np_ctx_aggregate_fwd(B("f").cptr(), B("out").cptr(), B("idx").cptr() if mode else None, T, nc, D, mode, None),
                  "ctx_aggregate_fwd")
    return Spec(call, bufs, {"out": (ref.double(), 1e-6)}, exact)


# ------------------------------------------------------------------------------------------------
# the route matrix
# ------------------------------------------------------------------------------------------------
HALO = "tapconv_halo_tma_kernel<{x3}, {nt}, {nb}>"
GATHER = "tapconv_umma_kernel<{x3}>"
SIMT = "tapconv_simt_kernel"
WH = "tapwgrad_halo_tma_kernel<{x3}>"
WH2 = "tapwgrad_halo_s2_kernel<{x3}>"
WU = "tapwgrad_umma_kernel<{x3}>"
WS = "tapwgrad_simt_kernel"
R32, R8, R1 = "reduce_partials_vec4_kernel<32>", "reduce_partials_vec4_kernel<8>", "reduce_partials_kernel"
COLSUM = "colsum_stage1"
GU = "gemm_umma_kernel<{x3}, {ak}, {bk}, {conv}>"
SPLITK = "splitk_epilogue_kernel"


def _x3(prec):
    return "true" if prec == "tf32x3" else "false"


def fwd_routes(route):
    """Expected kernels of a 64-channel convolution per precision; CUDA cores in fp32 mode."""
    out = {"fp32": {SIMT: 1}}
    for p in TC_PRECS:
        x3 = _x3(p)
        out[p] = {"halo": {HALO.format(x3=x3, nt=9, nb=6): 1},
                  "halo_s2": {HALO.format(x3=x3, nt=9, nb=3 if p == "tf32x3" else 6): 1},
                  "halo_skip": {HALO.format(x3=x3, nt=10, nb=4): 1},
                  "gather": {GATHER.format(x3=x3): 1},
                  "gather4": {GATHER.format(x3=x3): 4},
                  "simt": {SIMT: 1}}[route]
    if route == "gather4":
        out["fp32"] = {SIMT: 4}
    return out


def dgrad_routes(route, stride):
    out = fwd_routes(route)
    if stride == 2:
        out["fp32"] = {SIMT: 4}
    return out


def wgrad_routes(route, red, simt_red=None):
    """route kernel + the reduction of the weight partials and of the bias partials (red: reduce kernel by partial
    count); fp32 mode: CUDA-core kernel, its partials reduced with simt_red[0], the bias by colsum (stage 1 + the
    reduction named by simt_red[1])."""
    out = {}
    if simt_red is not None:
        out["fp32"] = collections.Counter({WS: 1, COLSUM: 1}) + collections.Counter([simt_red[0], simt_red[1]])
    for p in TC_PRECS:
        k = {"halo": WH, "halo_s2": WH2, "umma": WU, "simt": WS}[route].format(x3=_x3(p))
        if route == "simt":
            out[p] = out["fp32"]
        else:
            out[p] = collections.Counter({k: 1}) + collections.Counter([red, red])
    return out


def gemm_routes(ak, bk, conv=0, splitk=False, cuda_core=None):
    out = {"fp32": {cuda_core or "gemm_kernel": 1}}
    for p in TC_PRECS:
        out[p] = {GU.format(x3=_x3(p), ak=ak, bk=bk, conv=conv): 1}
        if splitk:
            out[p][SPLITK] = 1
    return out


# id: (builder, kwargs, expected kernels per precision, precisions)
CASES = {
    # --- conv_fwd 64 -> 64
    "fwd_s1_16x16_n3": (conv_fwd_spec, dict(N=3, H=16, W=16, stride=1, bits=True), fwd_routes("halo")),
    "fwd_s1_16x48": (conv_fwd_spec, dict(N=2, H=16, W=48, stride=1), fwd_routes("halo")),
    "fwd_s1_48x16": (conv_fwd_spec, dict(N=2, H=48, W=16, stride=1), fwd_routes("halo")),
    **{f"fwd_s1_16x8_n{n}": (conv_fwd_spec, dict(N=n, H=16, W=8, stride=1), fwd_routes("halo"))
       for n in (1, 148, 149, 297)},
    "fwd_s2_32x32": (conv_fwd_spec, dict(N=3, H=32, W=32, stride=2, bits=True), fwd_routes("halo_s2")),
    "fwd_s2_64x32": (conv_fwd_spec, dict(N=2, H=64, W=32, stride=2), fwd_routes("halo_s2")),
    "fwd_skip_16x16": (conv_fwd_spec, dict(N=3, H=16, W=16, stride=1, skip=True, bits=True), fwd_routes("halo_skip")),
    "fwd_skip_16x32": (conv_fwd_spec, dict(N=2, H=16, W=32, stride=1, skip=True), fwd_routes("halo_skip")),
    "fwd_gather_s2_16x16_n5": (conv_fwd_spec, dict(N=5, H=16, W=16, stride=2, bits=True), fwd_routes("gather")),
    "fwd_gather_s1_4x4_n5": (conv_fwd_spec, dict(N=5, H=4, W=4, stride=1), fwd_routes("gather")),
    "fwd_gather_s1_8x24": (conv_fwd_spec, dict(N=3, H=8, W=24, stride=1, skip=True), fwd_routes("gather")),
    "fwd_gather_s2_2x2_n129": (conv_fwd_spec, dict(N=129, H=2, W=2, stride=2), fwd_routes("gather")),
    "fwd_32to48": (conv_fwd_spec, dict(N=2, H=16, W=16, stride=2, cin=32, cout=48), fwd_routes("simt")),
    "fwd_48to64": (conv_fwd_spec, dict(N=2, H=8, W=12, stride=1, cin=48, cout=64), fwd_routes("simt")),
    # --- single-sign inputs (x >= 0, w >= 0) at a small and at the many-tiles size
    "fwd_s1_sign_16x16": (conv_fwd_spec, dict(N=3, H=16, W=16, stride=1, sign=True), fwd_routes("halo")),
    "fwd_s1_sign_n300_64": (conv_fwd_spec, dict(N=300, H=64, W=64, stride=1, sign=True), fwd_routes("halo")),
    "fwd_s2_sign_32x32": (conv_fwd_spec, dict(N=3, H=32, W=32, stride=2, sign=True), fwd_routes("halo_s2")),
    "fwd_s2_sign_n300_64": (conv_fwd_spec, dict(N=300, H=64, W=64, stride=2, sign=True), fwd_routes("halo_s2")),
    # --- conv_dgrad
    "dgrad_s1_16x16_src": (conv_dgrad_spec, dict(N=3, H=16, W=16, stride=1, mask="src"), dgrad_routes("halo", 1)),
    "dgrad_s1_16x16_bits": (conv_dgrad_spec, dict(N=3, H=16, W=16, stride=1, mask="bits"), dgrad_routes("halo", 1)),
    "dgrad_s2_32x32_src": (conv_dgrad_spec, dict(N=3, H=32, W=32, stride=2, mask="src"), dgrad_routes("halo", 2)),
    "dgrad_s2_32x32_bits": (conv_dgrad_spec, dict(N=3, H=32, W=32, stride=2, mask="bits"), dgrad_routes("halo", 2)),
    "dgrad_s2_skip_32x32": (conv_dgrad_spec, dict(N=3, H=32, W=32, stride=2, skip=True),
                            dgrad_routes("halo_skip", 2)),
    "dgrad_s2_skip_32x64": (conv_dgrad_spec, dict(N=2, H=32, W=64, stride=2, skip=True, mask="bits"),
                            dgrad_routes("halo_skip", 2)),
    "dgrad_gather_s2_16x16": (conv_dgrad_spec, dict(N=3, H=16, W=16, stride=2, skip=True, mask="src"),
                              dgrad_routes("gather4", 2)),
    "dgrad_gather_s1_8x8": (conv_dgrad_spec, dict(N=4, H=8, W=8, stride=1, mask="bits"), dgrad_routes("gather", 1)),
    "dgrad_gather_s1_8x24": (conv_dgrad_spec, dict(N=3, H=8, W=24, stride=1, mask="src"), dgrad_routes("gather", 1)),
    "dgrad_gather_s2_16x48": (conv_dgrad_spec, dict(N=2, H=16, W=48, stride=2), dgrad_routes("gather4", 2)),
    "dgrad_32to48": (conv_dgrad_spec, dict(N=2, H=16, W=16, stride=2, cin=32, cout=48), {p: {SIMT: 4} for p in PRECS}),
    "dgrad_48to64": (conv_dgrad_spec, dict(N=2, H=8, W=12, stride=1, cin=48, cout=64, mask="src"),
                     {p: {SIMT: 1} for p in PRECS}),
    # --- conv_wgrad
    "wgrad_s1_16x16_n3": (conv_wgrad_spec, dict(N=3, H=16, W=16, stride=1), wgrad_routes("halo", R1, (R1, R1))),
    "wgrad_s1_skip_16x16_n3": (conv_wgrad_spec, dict(N=3, H=16, W=16, stride=1, skip=True),
                               {p: wgrad_routes("halo", R1)[p] for p in TC_PRECS}),
    **{f"wgrad_s1_4x16_n{n}": (conv_wgrad_spec, dict(N=n, H=4, W=16, stride=1), wgrad_routes("halo", r, (R8, R8)))
       for n, r in ((148, R32), (149, R8), (297, R8))},
    "wgrad_s1_16x32": (conv_wgrad_spec, dict(N=2, H=16, W=32, stride=1), wgrad_routes("halo", R8, (R8, R1))),
    "wgrad_s1_32x16": (conv_wgrad_spec, dict(N=2, H=32, W=16, stride=1, skip=True),
                       {p: wgrad_routes("halo", R8)[p] for p in TC_PRECS}),
    "wgrad_s2_32x32": (conv_wgrad_spec, dict(N=3, H=32, W=32, stride=2), wgrad_routes("halo_s2", R8, (R1, R1))),
    **{f"wgrad_s2_4x32_n{n}": (conv_wgrad_spec, dict(N=n, H=4, W=32, stride=2), wgrad_routes("halo_s2", r, (R8, R8)))
       for n, r in ((148, R32), (149, R8))},
    "wgrad_umma_s1_8x8": (conv_wgrad_spec, dict(N=3, H=8, W=8, stride=1), wgrad_routes("umma", R1, (R1, R1))),
    "wgrad_umma_s1_8x8_n40": (conv_wgrad_spec, dict(N=40, H=8, W=8, stride=1), wgrad_routes("umma", R8, (R8, R1))),
    "wgrad_umma_1x1_s2": (conv_wgrad_spec, dict(N=5, H=16, W=16, stride=2, R=1), wgrad_routes("umma", R1, (R1, R1))),
    "wgrad_umma_s1_6x6_n5": (conv_wgrad_spec, dict(N=5, H=6, W=6, stride=1), wgrad_routes("umma", R1, (R1, R1))),
    "wgrad_32to48": (conv_wgrad_spec, dict(N=2, H=16, W=16, stride=2, cin=32, cout=48),
                     wgrad_routes("simt", None, (R1, R1))),
    "wgrad_48to64": (conv_wgrad_spec, dict(N=2, H=8, W=12, stride=1, cin=48, cout=64),
                     wgrad_routes("simt", None, (R1, R1))),
    "wgrad_s1_sign_16x16": (conv_wgrad_spec, dict(N=3, H=16, W=16, stride=1, sign=True),
                            wgrad_routes("halo", R1, (R1, R1))),
    "wgrad_s1_sign_n300_64": (conv_wgrad_spec, dict(N=300, H=64, W=64, stride=1, sign=True),
                              wgrad_routes("halo", R32)),
    "wgrad_s2_sign_32x32": (conv_wgrad_spec, dict(N=3, H=32, W=32, stride=2, sign=True),
                            wgrad_routes("halo_s2", R8, (R1, R1))),
    "wgrad_s2_sign_n300_64": (conv_wgrad_spec, dict(N=300, H=64, W=64, stride=2, sign=True),
                              wgrad_routes("halo_s2", R32)),
    # --- stems
    "stem_1_5_64_32x32": (stem_spec, dict(N=3, cin=1, H=32, W=32, R=5, cout=64, bits=True), None),
    "stem_1_5_64_32x64": (stem_spec, dict(N=2, cin=1, H=32, W=64, R=5, cout=64, bits=True), None),
    "stem_3_5_64": (stem_spec, dict(N=3, cin=3, H=16, W=16, R=5, cout=64), None),
    "stem_1_3_32": (stem_spec, dict(N=3, cin=1, H=32, W=32, R=3, cout=32), None),
    # --- gemm: the three dense-layer roles, tails, non-vector loads
    "gemm_fwd": (gemm_spec, dict(M=300, N=100, K=80, role="fwd", bias=True, act=1), gemm_routes("true", "true")),
    "gemm_dgrad": (gemm_spec, dict(M=300, N=80, K=100, role="dgrad"), gemm_routes("true", "false")),
    "gemm_wgrad": (gemm_spec, dict(M=100, N=80, K=200, role="wgrad"), gemm_routes("false", "false")),
    "gemm_fwd_m129": (gemm_spec, dict(M=129, N=64, K=64, role="fwd", bias=True), gemm_routes("true", "true")),
    "gemm_fwd_lda_odd": (gemm_spec, dict(M=200, N=64, K=64, role="fwd", pad_a=1), gemm_routes("true", "true")),
    "gemm_dgrad_lda_odd": (gemm_spec, dict(M=200, N=48, K=64, role="dgrad", pad_a=1), gemm_routes("true", "false")),
    "gemm_wgrad_lda_odd": (gemm_spec, dict(M=64, N=80, K=200, role="wgrad", pad_a=1), gemm_routes("false", "false")),
    # --- split-K
    "gemm_splitk2_bias_relu": (gemm_spec, dict(M=420, N=256, K=272, bias=True, act=1),
                               gemm_routes("true", "true", splitk=True)),
    "gemm_splitk11_tanh_beta_rowscale": (gemm_spec, dict(M=256, N=256, K=1419, bias=True, act=2, alpha=0.5, beta=1.0,
                                                         row_scale=True), gemm_routes("true", "true", splitk=True)),
    "gemm_sum_groups": (gemm_spec, dict(M=300, N=256, K=8 * 256, role="dgrad", groups=8),
                        {**gemm_routes("true", "false", splitk=True), "fp32": {"gemm_kernel": 8}}),
    "gemm_sum_groups_small": (gemm_spec, dict(M=64, N=96, K=3 * 64, role="dgrad", groups=3, bias=True, act=2),
                              {**gemm_routes("true", "false"), "fp32": {"gemm_kernel": 3}}),
    # --- CUDA-core GEMMs in the TF32 modes
    "gemm_skinny_n2": (gemm_spec, dict(M=37, N=2, K=256, bias=True),
                       {p: {"gemm_skinny_kernel": 1} for p in PRECS}),
    "gemm_small_n8": (gemm_spec, dict(M=100, N=8, K=32, role="dgrad", bias=True, act=1),
                      {p: {"gemm_kernel": 1} for p in PRECS}),
    # --- implicit convolution (tensor cores only)
    "gemm_conv_fwd_10x14": (gemm_spec, dict(M=5 * 5 * 7, N=48, K=9 * 32, conv=(1, 10, 14, 32, 5), bias=True),
                            {p: gemm_routes("true", "true", conv=1, splitk=True)[p] for p in TC_PRECS}),
    "gemm_conv_wgrad_10x14": (gemm_spec, dict(M=48, N=9 * 32, K=5 * 5 * 7, conv=(2, 10, 14, 32, 5)),
                              {p: gemm_routes("false", "false", conv=2)[p] for p in TC_PRECS}),
    "gemm_conv_fwd_sign_10x14": (gemm_spec, dict(M=5 * 5 * 7, N=48, K=9 * 32, conv=(1, 10, 14, 32, 5), sign=True),
                                 {p: gemm_routes("true", "true", conv=1, splitk=True)[p] for p in TC_PRECS}),
    "gemm_conv_wgrad_sign_10x14": (gemm_spec, dict(M=48, N=9 * 32, K=5 * 5 * 7, conv=(2, 10, 14, 32, 5), sign=True),
                                   {p: gemm_routes("false", "false", conv=2)[p] for p in TC_PRECS}),
    "gemm_conv_fwd_sign_n300_64": (gemm_spec, dict(M=300 * 32 * 32, N=48, K=9 * 32, conv=(1, 64, 64, 32, 300),
                                                   sign=True),
                                   {p: gemm_routes("true", "true", conv=1)[p] for p in TC_PRECS}),
    "gemm_conv_wgrad_sign_n300_64": (gemm_spec, dict(M=48, N=9 * 32, K=300 * 32 * 32, conv=(2, 64, 64, 32, 300),
                                                     sign=True),
                                     {p: gemm_routes("false", "false", conv=2, splitk=True)[p] for p in TC_PRECS}),
    # --- context aggregation: scalar kernel (D % 4 != 0, or a 4-B offset pointer) and the vector kernel
    "ctx_agg_mean_d37": (ctx_agg_spec, dict(T=6, nc=15, D=37, mode=0), {p: {"ctx_agg_fwd_kernel": 1} for p in PRECS}),
    "ctx_agg_max_d37": (ctx_agg_spec, dict(T=6, nc=15, D=37, mode=1), {p: {"ctx_agg_fwd_kernel": 1} for p in PRECS}),
    "ctx_agg_max_d256": (ctx_agg_spec, dict(T=6, nc=15, D=256, mode=1),
                         {p: {"ctx_agg_fwd_vec4_kernel": 1} for p in PRECS}),
}

STEM_ROUTES = {   # (Cin, R, Cout) -> expected per precision (forward + weight gradient in one case)
    (1, 5, 64): {"fp32": {"conv_small_fwd_kernel<1, 5>": 1, "conv_small_wgrad_stage1<1, 5>": 1, R8: 1},
                 **{p: {f"stem_fwd_umma_kernel<{_x3(p)}>": 1, f"stem_wgrad_umma_kernel<{_x3(p)}>": 1, R8: 1}
                    for p in TC_PRECS}},
    (3, 5, 64): {p: {"conv_small_fwd_kernel<3, 5>": 1, "conv_small_wgrad_stage1<3, 5>": 1, R8: 1} for p in PRECS},
    (1, 3, 32): {p: {"conv_small_fwd_kernel<1, 3>": 1, "conv_small_wgrad_stage1<1, 3>": 1, R32: 1} for p in PRECS},
}

# Single-sign inputs let the truncating fp32 accumulation of the tcgen05 kernels add up instead of cancel.  The 3x3
# stride-1 halo weight gradient at 1.2 M pixels misses the 4e-5 bar; tf32 at the same size measures the same error
# (5.5e-5), so it is the accumulator, not the operand split.
XFAIL = {("wgrad_s1_sign_n300_64", "tf32x3"):
         "halo weight gradient, x >= 0 and dy >= 0 over 1.2 M pixels: measured 5.56e-05 rel-L2 on a B200 against the "
         "4e-5 bar (fp32 accumulator truncation adds up over the pixel run of a TMEM block)"}


def _expected(case, prec):
    builder, kw, routes = CASES[case]
    if builder is stem_spec:
        routes = STEM_ROUTES[(kw["cin"], kw["R"], kw["cout"])]
    return routes.get(prec)


def _params():
    out = []
    for case, (builder, kw, routes) in CASES.items():
        big = kw.get("N", 0) >= 300 or kw.get("M", 0) >= 100_000 or kw.get("K", 0) >= 100_000
        for prec in PRECS:
            if _expected(case, prec) is None:
                continue
            marks = [pytest.mark.xfail(reason=XFAIL[case, prec], strict=True)] if (case, prec) in XFAIL else []
            for off in (("a256",) if big else ("a256", "a16")):
                out.append(pytest.param(case, prec, off, id=f"{case}-{prec}-{off}", marks=marks))
    return out


def _build(case, prec, off):
    builder, kw, _ = CASES[case]
    kw = dict(kw)
    if prec == "fp32" and "bits" in kw:
        kw["bits"] = False            # the packed gates are written by the tensor-core epilogues only
    return builder(prec, off=OFFSETS[off], **kw)


@pytest.mark.parametrize("case,prec,off", _params())
def test_route(case, prec, off):
    spec = _build(case, prec, off)
    res = run_case(spec, _expected(case, prec))
    rels = " ".join(f"{n}={v:.2e}" for n, v in res["rel"].items())
    print(f"\n[route] {case} {prec} {off}: {sorted(collections.Counter(res['kernels']).items())} rel-L2 {rels}")


@pytest.mark.parametrize("off", ["a4", "a8"])
def test_ctx_agg_unaligned_pointer_takes_the_scalar_kernel(off):
    """A feature pointer 4 or 8 bytes off 16-B alignment must route to the scalar kernel and still be right."""
    spec = ctx_agg_spec("fp32", 6, 15, 256, 1, off={"a4": 4, "a8": 8}[off])
    run_case(spec, {"ctx_agg_fwd_kernel": 1})


# ------------------------------------------------------------------------------------------------
# harness self-tests: each failure mode is reported
# ------------------------------------------------------------------------------------------------
def test_harness_reports_a_guard_overwrite():
    lib = _lib()
    out = Guarded("out", (1000,))

    def call():
        lib.check(lib.LIB.b200np_fill(out.cptr(), 1000, 1.0, None), "fill")
        out.bytes[out.off + out.nbytes] = 0            # one byte past the payload
    with pytest.raises(AssertionError, match="guard of 'out' overwritten"):
        run_case(Spec(call, {"out": out}, {}))


def test_harness_reports_an_unwritten_output():
    """N-1 images into an N-image payload: the last image is never written."""
    lib = _lib()
    spec = conv_fwd_spec("tf32x3", 4, 16, 16, 1)
    y = spec.bufs["y"]
    B = spec.bufs

    def call():
        lib.check(lib.LIB.b200np_conv_fwd(B["x"].cptr(), B["wf"].cptr(), B["b"].cptr(), y.cptr(), 3, 16, 16, 64, 64, 3,
                                          1, None, None, None, 0, 2, lib.ACT_RELU, PRECS["tf32x3"], None, None),
                  "conv_fwd")
    spec.call = call
    with pytest.raises(AssertionError, match="not fully written"):
        run_case(spec)


def test_harness_reports_a_kernel_that_did_not_run():
    lib = _lib()
    out = Guarded("out", (1000,))

    def call():
        lib.check(lib.LIB.b200np_fill(out.cptr(), 1000, 1.0, None), "fill")
    run_case(Spec(call, {"out": out}, {}), {"fill_kernel": 1})
    with pytest.raises(AssertionError, match="kernels: expected"):
        run_case(Spec(call, {"out": out}, {}), {"fill_kernel": 1, HALO.format(x3="true", nt=9, nb=6): 1})


def test_harness_reports_an_input_overrun_as_nan():
    """A read of one element past an input's end would pick up the NaN guard; here the host points the call one
    element into the trailing guard, which is what such a read amounts to."""
    lib = _lib()
    x = Guarded("in", (1000,), init=torch.ones(1000, device="cuda"))
    y = Guarded("out", (1000,))

    def call():
        lib.check(lib.LIB.b200np_scale_by_device_scalar(C.c_void_p(x.ptr + 4), x.cptr(), y.cptr(), 1000, None), "scale")
    with pytest.raises(AssertionError, match="NaN"):
        run_case(Spec(call, {"x": x, "y": y}, {}))


# ------------------------------------------------------------------------------------------------
# step coverage: every library kernel a training step launches is pinned by a case above or by this table
# ------------------------------------------------------------------------------------------------
SINGLE_KERNEL_ENTRY_POINTS = {   # kernel -> the existing test that covers it
    "adam_kernel": "test_gpu_ops.py::test_adam_matches_torch",
    "adam_tick_kernel": "test_gpu_models.py::test_fused_adam_training_steps_match_oracle",
    "act_bwd_kernel": "test_gpu_ops.py::test_elementwise_and_reductions",
    "axpy_kernel": "test_gpu_ops.py::test_elementwise_and_reductions",
    "fill_kernel": "test_gpu_ops.py::test_elementwise_and_reductions",
    "scale_dev_kernel": "test_gpu_ops.py::test_elementwise_and_reductions",
    "reduce_kernel": "test_gpu_ops.py::test_elementwise_and_reductions",
    "max_reduce_kernel": "test_gpu_ops.py::test_elementwise_and_reductions",
    "repeat_rows_kernel": "test_gpu_ops.py::test_elementwise_and_reductions",
    "repeat_rows_bwd_kernel": "test_gpu_ops.py::test_elementwise_and_reductions",
    "multi_copy_kernel": "test_gpu_models.py::test_model_matches_reference_and_oracle",
    "pack_weight_kernel": "test_gpu_ops.py::test_conv_block_ops",
    "amp2_flat_fwd_kernel": "test_gpu_ops.py::test_pools_and_flatten",
    "amp2_flat_bwd_kernel": "test_gpu_ops.py::test_pools_and_flatten",
    "nhwc_to_nchw_kernel": "test_gpu_ops.py::test_pools_and_flatten",
    "nchw_to_nhwc_kernel": "test_gpu_ops.py::test_pools_and_flatten",
    "maxpool2_fwd_kernel": "test_gpu_ops.py::test_pools_and_flatten",
    "maxpool2_fwd_vec4_kernel": "test_gpu_ops.py::test_pools_and_flatten",
    "maxpool2_bwd_kernel": "test_gpu_ops.py::test_pools_and_flatten",
    "maxpool2_bwd_vec4_kernel": "test_gpu_ops.py::test_pools_and_flatten",
    "ctx_agg_bwd_kernel": "test_gpu_ops.py::test_ctx_aggregate",
    "baco_fwd_kernel": "test_gpu_ops.py::test_baco_aggregation",
    "baco_bwd_kernel": "test_gpu_ops.py::test_baco_aggregation",
    "loss_kernel": "test_gpu_ops.py::test_loss_large_batches",
    "loss_multi_kernel": "test_gpu_ops.py::test_loss_large_batches",
    "loss_multi_vec_kernel": "test_gpu_ops.py::test_loss_large_batches",
    "favor_rowstats_kernel": "test_gpu_ops.py::test_favor_attention_fwd_bwd",
    "favor_attn_fwd_kernel": "test_gpu_ops.py::test_favor_attention_fwd_bwd",
    "favor_attn_bwd_kernel": "test_gpu_ops.py::test_favor_attention_fwd_bwd",
    "favor_key_fixup_kernel": "test_gpu_ops.py::test_favor_attention_fwd_bwd",
    "im2col_small_kernel": "test_gpu_ops.py::test_small_cin_im2col_gemm_stem",
    "col2im3x3s2_tapmajor_kernel": "test_gpu_ops.py::test_implicit_conv_gemm",
    "conv_weight_tapmajor_kernel": "test_gpu_ops.py::test_implicit_conv_gemm",
    "gather_images_u8_kernel": "test_sampler.py::test_gather_images_u8_rgb_and_full_size",
}


def _library_kernel_names():
    """Base names of every __global__ function in the library sources."""
    csrc = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                        "what-matters-for-meta-learning_b200", "csrc")
    names = set()
    pat = re.compile(r"__global__\s+(?:void\s+)?(?:__launch_bounds__\([^)]*\)\s+)?(?:void\s+)?(\w+)\s*\(")
    for path in glob.glob(os.path.join(csrc, "*.cu")):
        with open(path) as f:
            names.update(pat.findall(f.read()))
    return names


def _route_kernels():
    out = set()
    for case in CASES:
        for prec in PRECS:
            e = _expected(case, prec)
            if e:
                out.update(e)
    return out


def _step_kernels(model_name, prec):
    import bench
    from b200np import engine
    from b200np.optim import FlatParams, FusedAdam
    from oracle import synth
    from trainer.losses import LossFunc
    engine.set_precision(prec)
    task, _, _, _, T, views = bench.MODELS[model_name]
    nc = 15
    nt = views - nc if task == "distractor" else 15
    model = getattr(importlib.import_module(f"networks.{model_name}"), model_name)(
        bench.make_cfg(T, "cuda", model_name)).to("cuda")
    flat = FlatParams(model)
    opt = FusedAdam(flat, lr=1e-4)
    lossf = LossFunc("mse", task)
    b = [torch.from_numpy(a).cuda() for a in synth.task_batch(task, T, nc, nt, seed=1)]

    def step():
        opt.zero_grad()
        mu, _, _ = model(b[0], b[1], b[2])
        lossf.calc_loss(mu, None, b[3]).backward()
        opt.step()
    step()
    torch.cuda.synchronize()
    return launched(step)


_reached = set()
# tf32 takes the 6-slot weight ring wherever tf32x3 takes 3 (its planes need half the shared memory), and no form needs
# more than 3 slots' worth of room in tf32
NEVER_SELECTED = "tapconv_halo_tma_kernel<false, 9, 3>"


@pytest.mark.parametrize("prec", TC_PRECS)
@pytest.mark.parametrize("model_name", ["ANPDistractor", "CNPDistractor", "ANP", "CondNeuralProcess", "CNPShapeNet1D",
                                        "ANPShapeNet1D"])
def test_step_launches_only_pinned_kernels(model_name, prec):
    import bench
    assert model_name in bench.MODELS
    lib_names = _library_kernel_names()
    claimed = _route_kernels() | set(SINGLE_KERNEL_ENTRY_POINTS)
    ks = _step_kernels(model_name, prec)
    ours = {k for k in ks if k.partition("<")[0] in lib_names}
    _reached.update(ours)
    unclaimed = sorted(ours - claimed)
    print(f"\n[step] {model_name} {prec}: {len(ks)} launches, library kernels {sorted(ours)}")
    assert not unclaimed, f"library kernels no route case or entry-point test pins: {unclaimed}"


def test_report_route_kernels_no_step_reached():
    """Listing only (run after the step tests): kernels a route case pins that no benchmarked step launches."""
    if not _reached:
        pytest.skip("no step test ran in this session")
    print("\n[unreached] " + ", ".join(sorted(_route_kernels() - _reached)))
    print(f"[unselected] {NEVER_SELECTED}: compiled, but no convolution form selects it")
