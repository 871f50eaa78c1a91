"""Autograd functions over the C ABI (include/galerkin_b200.h).

Every function here hands raw device pointers, sizes and the current CUDA stream to
libgalerkin_b200.so; PyTorch is used for memory (torch.empty from the caching allocator),
streams and the autograd graph only.  Backward runs on PyTorch's autograd thread; the
library is re-entrant and takes the device ordinal on every call.
"""
import contextlib
import ctypes
import os
import math
import threading
import weakref

import torch

from . import _lib
from ._lib import HeadOperand, check, ptr, stream_of, workspace, require_cuda_f32

ACT = {"none": 0, None: 0, "identity": 0, "relu": 1, "silu": 2}

# GEMM arithmetic (fp32 storage everywhere):
#   "x3"   (default) error-compensated split: the fused encoder-layer kernels run every product as three bf16 tensor-core
#          products (a_hi b_hi + a_hi b_lo + a_lo b_hi, fp32 accumulate: ~2^-17 per product); weight-gradient GEMMs
#          (sums over all tokens, where TF32 rounding averages out: measured 5e-6) run single-pass TF32 on tcgen05;
#          anything not covered by a fused kernel falls back to exact fp32 FMAs.  Meets the stated fp32 parity
#          tolerances (DESIGN.md section 1).
#   "tf32" every GEMM single-pass TF32 on tcgen05 (fastest unfused path; ~1e-2 gradient error through 10 layers)
#   "fp32" exact-fp32 SIMT FMAs everywhere (the precise mode used by the tight parity tests).
_PRECISION = "x3"


def set_precision(mode):
    """'x3' (default: bf16x3 fused kernels + TF32 weight gradients), 'tf32' or 'fp32' (exact SIMT path)."""
    global _PRECISION
    assert mode in ("x3", "tf32", "fp32")
    _PRECISION = mode
    # the stock cuDNN 3x3 convolutions of the interpolation scalers (out of scope, SURVEY 8f-1) follow the mode:
    # TF32 only in 'tf32' mode (torch's default would be TF32 always)
    torch.backends.cudnn.allow_tf32 = mode == "tf32"


def get_precision():
    return _PRECISION


torch.backends.cudnn.allow_tf32 = _PRECISION == "tf32"

_SPLIT_MIN_FLOPS = 0.5e9   # measured: C5's 0.15 GFLOP GEMMs lose, C3's 1.3 win
_seed_lock = threading.Lock()
_seed_counter = 0


def _rank():
    try:
        import torch.distributed as dist
        return dist.get_rank() if dist.is_available() and dist.is_initialized() else 0
    except Exception:
        return 0


def next_seed():
    """63-bit Philox key for one fused-dropout site: derived from torch's seed, the distributed rank (identically seeded
    data-parallel replicas still draw different masks on their shards) and a process-local call counter -- deterministic
    under torch.manual_seed."""
    global _seed_counter
    with _seed_lock:
        _seed_counter += 1
        c = _seed_counter + 0x51ED270B * _rank()
    # 63 bits: the value travels through autograd.Function arguments, which profilers convert to int64
    return (torch.initial_seed() * 0x9E3779B97F4A7C15 + c * 0xD1B54A32D192ED03) & 0x7FFFFFFFFFFFFFFF


def _dev(t):
    return t.device.index if t.device.index is not None else torch.cuda.current_device()


_rng_step = None


def rng_step_counter(device=None):
    """Device-side int64 step counter added to every fused-dropout seed (one per process/GPU).
    `advance_rng()` bumps it with a tiny kernel, which -- unlike a Python-side seed -- still works when
    the whole step is replayed from a CUDA graph (see graphs.py)."""
    global _rng_step
    if _rng_step is None:
        _rng_step = torch.zeros(1, dtype=torch.int64, device=device or torch.device("cuda", torch.cuda.current_device()))
        check(_lib.load().gb200_set_rng_offset_ptr(_rng_step.data_ptr()), "gb200_set_rng_offset_ptr")
    return _rng_step


def advance_rng():
    rng_step_counter().add_(0x9E3779B1)


def get_rng_state():
    """(call counter, device step counter) of the fused-dropout streams -- put it in checkpoints next to torch's RNG state"""
    return dict(seed_counter=_seed_counter, step=int(rng_step_counter().item()) if _rng_step is not None else None)


def set_rng_state(state):
    global _seed_counter
    _seed_counter = int(state["seed_counter"])
    if state.get("step") is not None:
        rng_step_counter().fill_(int(state["step"]))


class Profiler:
    """Optional per-launch CUDA-event attribution (bench.py's roofline pass).  When enabled every
    native launch is bracketed by two events on the launching stream and tagged with its
    ALGORITHMIC flops / bytes (DESIGN.md section 4)."""
    enabled = False
    records = []          # (family, start_event, end_event, flops, bytes)

    @classmethod
    def reset(cls):
        cls.records = []

    @classmethod
    def summary(cls):
        agg = {}
        for fam, s, e, fl, by in cls.records:
            a = agg.setdefault(fam, dict(launches=0, ms=0.0, flops=0.0, bytes=0.0))
            a["launches"] += 1
            a["ms"] += s.elapsed_time(e)
            a["flops"] += fl
            a["bytes"] += by
        return agg


def _launch(family, flops, nbytes, fn, *args):
    if Profiler.enabled:
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        rc = fn(*args)
        e.record()
        Profiler.records.append((family, s, e, float(flops), float(nbytes)))
    else:
        rc = fn(*args)
    if rc != 0:
        check(rc, family)


# ------------------------------------------------------------------------------------------
# backward fork/join: weight- and bias-gradient launches leave the critical path
# ------------------------------------------------------------------------------------------
_BWD_STREAMS = os.environ.get("GB200_BWD_STREAMS", "1") != "0"
_side_streams = {}


def set_backward_streams(on):
    """Run the parameter-gradient launches of each backward (dW GEMM + split-K reduce, bias column sums) on side
    streams, concurrently with the input-gradient GEMM that the next backward node is waiting for.  Every one of
    these kernels is a single latency-bound wave at the shipped sizes, so they overlap almost freely; inside a
    captured step the fork/join becomes parallel branches of the CUDA graph."""
    global _BWD_STREAMS
    _BWD_STREAMS = bool(on)


def _weak(t):
    """weak reference to an optional parameter tensor (autograd contexts must not keep non-saved tensors alive)"""
    return (lambda: None) if t is None else weakref.ref(t)


class _Fork:
    """`with fork.side(i):` enqueues on side stream i (which first waits, on every entry, for everything enqueued on
    the launching stream so far); `join()` makes the launching stream wait for the side work.  Outputs must be allocated BEFORE
    entering a side context (they then belong to the launching stream's allocator pool, and the join orders every
    later use after the side-stream writes); scratch allocated inside stays on the side stream."""

    def __init__(self, like):
        self.device = like.device
        self.main = torch.cuda.current_stream(self.device)
        self.used = []

    def side(self, i):
        if not _BWD_STREAMS:
            return contextlib.nullcontext()
        # one pool per launching stream: concurrent micro-batch chains (graphs.py batch_streams) must not share side
        # streams, or their joins would serialise the chains
        pool = _side_streams.setdefault((self.device.index, self.main.cuda_stream), [])
        while len(pool) <= i:
            pool.append(torch.cuda.Stream(device=self.device))
        s = pool[i]
        s.wait_stream(self.main)       # on EVERY entry: later side work may consume later launching-stream results
        if s not in self.used:
            self.used.append(s)
        return torch.cuda.stream(s)

    def join(self):
        for s in self.used:
            self.main.wait_stream(s)
        self.used = []

    def join_at_end_of_backward(self, keepalive):
        """Do not wait now: the launching stream joins the side streams when the whole backward pass has been enqueued
        (autograd engine callback), so weight-gradient GEMMs of layer l overlap the input-gradient chain of layers
        l-1, l-2, ...  `keepalive`: every tensor the side work reads or writes -- held until the join so the caching
        allocator cannot hand their memory to later launches of the same pass."""
        global _join_queued
        if not self.used:
            return
        with _seed_lock:
            _pending_joins.append((self.main, list(self.used), keepalive))
            queue = not _join_queued
            _join_queued = True
        self.used = []
        if queue:
            torch.autograd.Variable._execution_engine.queue_callback(_join_pending)


_aux_streams = {}


def aux_stream(device):
    """one auxiliary stream per device for work that is independent of the critical path (parameter packing)"""
    key = device.index if device.index is not None else torch.cuda.current_device()
    if key not in _aux_streams:
        _aux_streams[key] = torch.cuda.Stream(device=device)
    return _aux_streams[key]


_pending_joins = []
_join_queued = False
_DEFER_WGRAD_JOIN = True      # graphs.GraphedStep clears it for concurrent micro-batch chains


def _join_pending():
    global _join_queued
    with _seed_lock:
        items = list(_pending_joins)
        _pending_joins.clear()
        _join_queued = False
    for main, streams, _keep in items:
        for st in streams:
            main.wait_stream(st)


def _note_use(*params):
    """Forward bookkeeping for _finish_fork: how many autograd nodes of the graph being built use each parameter."""
    if not torch.is_grad_enabled():
        return
    for p in params:
        if p is not None and p.requires_grad:
            p._gb200_pending = getattr(p, "_gb200_pending", 0) + 1
            p._gb200_total = getattr(p, "_gb200_total", 0) + 1


def _single_use(params):
    """Backward: True when every parameter feeds exactly ONE node of this graph and has no gradient yet -- only then does
    autograd adopt the gradient tensor as it is.  A parameter used several times (a rollout applying the model repeatedly) or
    with an existing .grad is summed by the engine on the launching stream, which must then see finished side-stream work."""
    ok = True
    for p in params:
        if p is None:
            continue
        if not p.is_leaf or getattr(p, "_gb200_total", 1) > 1 or p.grad is not None:
            ok = False          # (a non-leaf "parameter", e.g. a packed weight, is consumed by the next node right away)
        pend = getattr(p, "_gb200_pending", 1) - 1
        p._gb200_pending = max(pend, 0)
        if pend <= 0:
            p._gb200_total = 0
    return ok


def _finish_fork(fork, params, keepalive):
    """End of a backward node whose parameter gradients were launched on side streams: normally the launching stream joins
    them only when the whole backward pass has been enqueued (they then overlap every later node instead of the rest of
    this one).  That needs autograd to ADOPT the gradient tensors (`p.grad is None`: no accumulation kernel on the
    launching stream before the side stream has written them) -- otherwise, or with _DEFER_WGRAD_JOIN cleared, join now.
    `keepalive`: the tensors the side work reads (not its outputs: a second reference would make autograd copy them)."""
    if _single_use(params) and _DEFER_WGRAD_JOIN:
        fork.join_at_end_of_backward(keepalive)
    else:
        fork.join()


# ------------------------------------------------------------------------------------------
# raw launches
# ------------------------------------------------------------------------------------------
def gemm(A, B, C, M, N, K, *, lda, ldb, ldc, transA=False, transB=False, alpha=1.0, bias=None, act=0,
         zout=None, ldz=0, drop_p=0.0, seed=0, residual=None, ldr=0, rscale=1.0, accumulate=False,
         ksplit=None, a_off=0, b_off=0, c_off=0, gate=None, ldg=0, gate_act=0, wgrad=False):
    """C = R + rscale*drop(act(alpha*op(A).op(B)+bias)); offsets are in floats.
    gate (with gate_act relu|silu): C = rscale*drop((alpha*op(A).op(B)) * act'(gate)) -- no bias/act/residual.
    wgrad: a weight-gradient GEMM (contraction over all tokens): single-pass TF32 also in 'x3' mode."""
    lib = _lib.load()
    pa, pb = ptr(A) + 4 * a_off, ptr(B) + 4 * b_off
    nbytes = 4.0 * (M * K + K * N + M * N * (1 + (residual is not None) + (zout is not None) + (gate is not None)))
    lay = ("t" if transA else "n") + ("t" if transB else "n")
    use_tc = _PRECISION in ("tf32", "x3") and lib.gb200_gemm_tc_supported(pa, lda, pb, ldb, M, N, K)
    # forward / input-gradient GEMM outside the fused kernels in 'x3' mode: 3xTF32
    split = use_tc and _PRECISION == "x3" and not wgrad
    if split and 2.0 * M * N * K < _SPLIT_MIN_FLOPS:   # small problems: the exact SIMT kernel has the shorter fixed latency
        use_tc = split = False
    if gate is not None:
        assert bias is None and act == 0 and zout is None and residual is None and not accumulate
        if ksplit is None:
            ksplit = lib.gb200_gemm_tc_suggest_ksplit(M, N, K) if use_tc else lib.gb200_gemm_suggest_ksplit(M, N, K, 1)
        ws_bytes = ksplit * M * N * 4 if ksplit > 1 else 0
        ws = workspace(ws_bytes, C)
        args = (_dev(C), pa, lda, int(transA), pb, ldb, int(transB), ptr(C) + 4 * c_off, ldc, M, N, K, alpha, drop_p, seed,
                rscale, ptr(gate), ldg, gate_act, ksplit, ptr(ws), ws_bytes)
        if use_tc:
            _launch("gemm_tc_" + lay, 2.0 * M * N * K, nbytes, lib.gb200_gemm_tc_gated, *args, int(split), stream_of(C))
        else:
            _launch("gemm_simt_" + lay, 2.0 * M * N * K, nbytes, lib.gb200_gemm_gated, *args, stream_of(C))
        return
    if use_tc:
        if ksplit is None:
            ksplit = lib.gb200_gemm_tc_suggest_ksplit(M, N, K)
        ws_bytes = ksplit * M * N * 4 if ksplit > 1 else 0
        ws = workspace(ws_bytes, C)
        _launch("gemm_tc_" + lay, 2.0 * M * N * K, nbytes, lib.gb200_gemm_tc, _dev(C), pa, lda, int(transA), pb,
                ldb, int(transB), ptr(C) + 4 * c_off, ldc, M, N, K, alpha, ptr(bias), act, ptr(zout), ldz, drop_p,
                seed, ptr(residual), ldr, rscale, int(accumulate), ksplit, ptr(ws), ws_bytes, int(split), stream_of(C))
        return
    if ksplit is None:
        ksplit = lib.gb200_gemm_suggest_ksplit(M, N, K, 1)
    ws_bytes = lib.gb200_gemm_workspace_bytes(M, N, K, 1, ksplit)
    ws = workspace(ws_bytes, C)
    _launch("gemm_simt_" + lay, 2.0 * M * N * K, nbytes, lib.gb200_gemm, _dev(C), pa, lda, int(transA), pb, ldb,
            int(transB), ptr(C) + 4 * c_off, ldc, M, N, K, 1, 0, 0, 0, alpha, ptr(bias), act, ptr(zout), ldz,
            drop_p, seed, ptr(residual), ldr, rscale, int(accumulate), ksplit, ptr(ws), ws_bytes, stream_of(C))


def wgrad_group(problems, T):
    """[(G (T, M) view, M, ldg, X (T, N), N, dW (M, N)), ...] (at most 6): dW = G^T X for each, one tcgen05 TF32 split-K launch
    and one deterministic reduction for the whole group (gb200_gemm_tc_wgrad_group)."""
    lib = _lib.load()
    n = len(problems)
    arr = (_lib.WgradProblem * n)()
    flops = nbytes = 0.0
    for i, (G_, M, ldg, X_, N, dW) in enumerate(problems):
        arr[i].G, arr[i].ldg, arr[i].X, arr[i].ldx = G_.data_ptr(), ldg, ptr(X_), N
        arr[i].dW, arr[i].ldw, arr[i].M, arr[i].N, arr[i].T = ptr(dW), N, M, N, T
        flops += 2.0 * T * M * N
        nbytes += 4.0 * (T * (M + N) + M * N)
    like = problems[0][0]
    wsb = lib.gb200_gemm_tc_wgrad_group_workspace_bytes(n, arr)
    ws = workspace(wsb, like)
    _launch("gemm_tc_tn", flops, nbytes, lib.gb200_gemm_tc_wgrad_group, _dev(like), n, arr, ptr(ws), wsb, stream_of(like))


def colsum(X, M, N, ld, out, *, x_off=0, scale=1.0, accumulate=False):
    lib = _lib.load()
    ws_bytes = lib.gb200_colsum_workspace_bytes(M, N)
    ws = workspace(ws_bytes, X)
    _launch("colsum", M * N, 4.0 * M * N, lib.gb200_colsum, _dev(X), ptr(X) + 4 * x_off, ld, M, N, scale,
            int(accumulate), ptr(out), ptr(ws), ws_bytes, stream_of(X))


def epilogue_bwd(dy, M, N, *, z=None, y=None, act=0, rscale=1.0, drop_p=0.0, seed=0):
    g = torch.empty((M, N), dtype=torch.float32, device=dy.device)
    _launch("epilogue_bwd", 4.0 * M * N, 4.0 * M * N * (2 + (act != 0)), _lib.load().gb200_epilogue_bwd,
            _dev(dy), ptr(dy), N, ptr(z), N, ptr(y), N, ptr(g), N, M, N, act, rscale, drop_p, seed,
            stream_of(dy))
    return g


# ------------------------------------------------------------------------------------------
# parameter packing
# ------------------------------------------------------------------------------------------
class _PackFn(torch.autograd.Function):
    """flat = concat(t.reshape(-1) for t in tensors) in ONE kernel; backward hands each parameter a view of the
    incoming flat gradient (no kernels)."""

    @staticmethod
    def forward(ctx, *tensors):
        require_cuda_f32(*tensors)
        import ctypes
        n = len(tensors)
        ts = [t if t.is_contiguous() else t.contiguous() for t in tensors]
        sizes = [t.numel() for t in ts]
        flat = torch.empty(sum(sizes), dtype=torch.float32, device=ts[0].device)
        srcs = (ctypes.c_void_p * n)(*[t.data_ptr() for t in ts])
        szs = (ctypes.c_longlong * n)(*sizes)
        _launch("pack", 0.0, 8.0 * sum(sizes), _lib.load().gb200_pack, _dev(flat), ptr(flat), srcs, szs, n,
                stream_of(flat))
        ctx.shapes = [t.shape for t in tensors]
        ctx.sizes = sizes
        return flat

    @staticmethod
    def backward(ctx, g):
        out, off = [], 0
        for shape, n in zip(ctx.shapes, ctx.sizes):
            out.append(g[off:off + n].view(shape))
            off += n
        return tuple(out)


def pack(tensors):
    return _PackFn.apply(*tensors)


# ------------------------------------------------------------------------------------------
# Linear (+bias, activation, fused dropout, signed residual)
# ------------------------------------------------------------------------------------------
class _LinearFn(torch.autograd.Function):
    """y = residual + rscale * dropout_p(act(x @ W^T + b));  x: (M, K), W: (N, K)."""

    @staticmethod
    def forward(ctx, x, weight, bias, residual, act, rscale, drop_p, seed):
        require_cuda_f32(x, weight, bias, residual)
        M, K = x.shape
        N = weight.shape[0]
        y = torch.empty((M, N), dtype=torch.float32, device=x.device)
        # backward needs act'(z): SiLU always from z; ReLU from the stored output unless a residual
        # was folded into it
        # (a ReLU gate read from the stored output y = rscale * drop(relu(z)) needs rscale > 0)
        needs_grad = x.requires_grad or weight.requires_grad or (bias is not None and bias.requires_grad)
        need_z = (act == ACT["silu"] or (act == ACT["relu"] and (residual is not None or rscale <= 0.0))) and needs_grad
        z = torch.empty_like(y) if need_z else None
        gemm(x, weight, y, M, N, K, lda=K, ldb=K, ldc=N, transB=True, bias=bias, act=act, zout=z, ldz=N,
             drop_p=drop_p, seed=seed, residual=residual, ldr=N, rscale=rscale)
        ctx.save_for_backward(x, weight, z, y if (act == ACT["relu"] and z is None) else None)
        ctx.cfg = (act, rscale, drop_p, seed, bias is not None, residual is not None)
        ctx.bias_ref = _weak(bias)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, weight, z, y = ctx.saved_tensors
        act, rscale, drop_p, seed, has_bias, has_res = ctx.cfg
        dy = dy.contiguous()
        M, K = x.shape
        N = weight.shape[0]
        dx = dw = db = None
        want_db = has_bias and ctx.needs_input_grad[2]
        if act != 0 or drop_p > 0.0 or rscale != 1.0:
            if want_db:      # one pass: g and its column sums
                lib = _lib.load()
                g = torch.empty((M, N), dtype=torch.float32, device=dy.device)
                db = torch.empty(N, dtype=torch.float32, device=dy.device)
                wsb = lib.gb200_epilogue_bwd_bias_workspace_bytes(M, N)
                ws = workspace(wsb, dy)
                _launch("epilogue_bwd_bias", 5.0 * M * N, 4.0 * M * N * (2 + (act != 0)), lib.gb200_epilogue_bwd_bias,
                        _dev(dy), ptr(dy), N, ptr(z), N, ptr(y), N, ptr(g), N, M, N, act, rscale, drop_p, seed, ptr(db),
                        ptr(ws), wsb, stream_of(dy))
                want_db = False
            else:
                g = epilogue_bwd(dy, M, N, z=z, y=y, act=act, rscale=rscale, drop_p=drop_p, seed=seed)
        else:
            g = dy
        fork = _Fork(g)
        if ctx.needs_input_grad[1]:
            dw = torch.empty_like(weight)
            with fork.side(0):
                gemm(g, x, dw, N, K, M, lda=N, ldb=K, ldc=K, transA=True, wgrad=True)
        if want_db:
            db = torch.empty(N, dtype=torch.float32, device=x.device)
            with fork.side(1):
                colsum(g, M, N, N, db)
        if ctx.needs_input_grad[0]:
            dx = torch.empty_like(x)
            gemm(g, weight, dx, M, K, N, lda=N, ldb=K, ldc=K)
        _finish_fork(fork, (weight, ctx.bias_ref()), (g, x))
        dres = dy if (has_res and ctx.needs_input_grad[3]) else None
        return dx, dw, db, dres, None, None, None, None


class _MLP2Fn(torch.autograd.Function):
    """y = [x +] rscale * drop_p2( drop_p1(act(x W1^T + b1)) W2^T + b2 )  -- FeedForward (libs/layers.py:979-987) with
    the encoder's residual + dropout2 (libs/model.py:132), and the regressor head Linear-act-Linear
    (libs/model.py:595-600, 629).  One autograd node, so backward is three launches on the critical path:
        g2 = dy * mask2 * rscale            (skipped when p2 = 0 and rscale = 1)
        g1 = (g2 W2) * act'(z1) * mask1     (gated GEMM epilogue: no elementwise pass between the layers)
        dx = dy + g1 W1                     (the shortcut's gradient rides in the last GEMM's epilogue)
    while dW2, dW1, db1 (and db2) run on the side streams."""

    @staticmethod
    def forward(ctx, x, w1, b1, w2, b2, act, p1, seed1, p2, seed2, rscale, shortcut):
        require_cuda_f32(x, w1, b1, w2, b2)
        M, K = x.shape
        N1, N2 = w1.shape[0], w2.shape[0]
        h = torch.empty((M, N1), dtype=torch.float32, device=x.device)
        need_grad = x.requires_grad or w1.requires_grad or w2.requires_grad or \
            (b1 is not None and b1.requires_grad) or (b2 is not None and b2.requires_grad)
        z1 = torch.empty_like(h) if (act == ACT["silu"] and need_grad) else None
        gemm(x, w1, h, M, N1, K, lda=K, ldb=K, ldc=N1, transB=True, bias=b1, act=act, zout=z1, ldz=N1, drop_p=p1,
             seed=seed1)
        y = torch.empty((M, N2), dtype=torch.float32, device=x.device)
        gemm(h, w2, y, M, N2, N1, lda=N1, ldb=N1, ldc=N2, transB=True, bias=b2, drop_p=p2, seed=seed2,
             residual=x if shortcut else None, ldr=K, rscale=rscale)
        ctx.save_for_backward(x, w1, w2, h, z1)
        ctx.cfg = (act, p1, seed1, p2, seed2, rscale, shortcut, b1 is not None, b2 is not None)
        ctx.bias_refs = (_weak(b1), _weak(b2))
        return y

    @staticmethod
    def backward(ctx, dy):
        x, w1, w2, h, z1 = ctx.saved_tensors
        act, p1, seed1, p2, seed2, rscale, shortcut, has_b1, has_b2 = ctx.cfg
        dy = dy.contiguous()
        M, K = x.shape
        N1, N2 = w1.shape[0], w2.shape[0]
        lib = _lib.load()
        dx = dw1 = db1 = dw2 = db2 = None
        want_db2 = has_b2 and ctx.needs_input_grad[4]
        fork = _Fork(dy)
        if p2 > 0.0 or rscale != 1.0:
            if want_db2:
                g2 = torch.empty_like(dy)
                db2 = torch.empty(N2, dtype=torch.float32, device=dy.device)
                wsb = lib.gb200_epilogue_bwd_bias_workspace_bytes(M, N2)
                ws = workspace(wsb, dy)
                _launch("epilogue_bwd_bias", 5.0 * M * N2, 8.0 * M * N2, lib.gb200_epilogue_bwd_bias, _dev(dy), ptr(dy),
                        N2, None, N2, None, N2, ptr(g2), N2, M, N2, 0, rscale, p2, seed2, ptr(db2), ptr(ws), wsb,
                        stream_of(dy))
            else:
                g2 = epilogue_bwd(dy, M, N2, rscale=rscale, drop_p=p2, seed=seed2)
        else:
            g2 = dy
            if want_db2:
                db2 = torch.empty(N2, dtype=torch.float32, device=dy.device)
                with fork.side(1):
                    colsum(g2, M, N2, N2, db2)
        if ctx.needs_input_grad[3]:
            dw2 = torch.empty_like(w2)
            with fork.side(0):
                gemm(g2, h, dw2, N2, N1, M, lda=N2, ldb=N1, ldc=N1, transA=True, wgrad=True)
        # g1 = (g2 W2) * act'(.) * mask1: ReLU gates on the stored (post-dropout) output, SiLU on the pre-activation
        g1 = torch.empty_like(h)
        if act == ACT["none"] and p1 == 0.0:
            gemm(g2, w2, g1, M, N1, N2, lda=N2, ldb=N1, ldc=N1)
        elif act == ACT["none"]:
            # dropout only: gate on "kept" via a ReLU gate is wrong for negative values -> plain GEMM + mask pass
            gemm(g2, w2, g1, M, N1, N2, lda=N2, ldb=N1, ldc=N1)
            g1 = epilogue_bwd(g1, M, N1, drop_p=p1, seed=seed1)
        else:
            gemm(g2, w2, g1, M, N1, N2, lda=N2, ldb=N1, ldc=N1, drop_p=p1, seed=seed1,
                 gate=h if act == ACT["relu"] else z1, ldg=N1, gate_act=act)
        if ctx.needs_input_grad[1]:
            dw1 = torch.empty_like(w1)
            with fork.side(0):
                gemm(g1, x, dw1, N1, K, M, lda=N1, ldb=K, ldc=K, transA=True, wgrad=True)
        if has_b1 and ctx.needs_input_grad[2]:
            db1 = torch.empty(N1, dtype=torch.float32, device=dy.device)
            with fork.side(1):
                colsum(g1, M, N1, N1, db1)
        if ctx.needs_input_grad[0]:
            dx = torch.empty_like(x)
            gemm(g1, w1, dx, M, K, N1, lda=N1, ldb=K, ldc=K, residual=dy if shortcut else None, ldr=N2)
        _finish_fork(fork, (w1, w2, ctx.bias_refs[0](), ctx.bias_refs[1]()), (dy, g2, g1, h, x))
        return dx, dw1, db1, dw2, db2, None, None, None, None, None, None, None


def mlp2(x, w1, b1, w2, b2, *, act="relu", drop_p1=0.0, drop_p2=0.0, rscale=1.0, shortcut=False):
    """Linear -> act -> dropout -> Linear [-> dropout -> rscale -> + x]; any leading shape."""
    lead = x.shape[:-1]
    x2 = x.reshape(-1, x.shape[-1]).contiguous()
    if shortcut:
        assert w2.shape[0] == x2.shape[1]
    seed1 = next_seed() if drop_p1 > 0.0 else 0
    seed2 = next_seed() if drop_p2 > 0.0 else 0
    _note_use(w1, w2, b1, b2)
    y = _MLP2Fn.apply(x2, w1, b1, w2, b2, ACT[act], float(drop_p1), seed1, float(drop_p2), seed2, float(rscale),
                      bool(shortcut))
    return y.reshape(*lead, w2.shape[0])


def linear(x, weight, bias=None, *, act="none", residual=None, rscale=1.0, drop_p=0.0):
    """nn.Linear over the last dimension with the fused epilogue; any leading shape."""
    lead = x.shape[:-1]
    x2 = x.reshape(-1, x.shape[-1]).contiguous()
    r2 = None if residual is None else residual.reshape(-1, weight.shape[0]).contiguous()
    seed = next_seed() if drop_p > 0.0 else 0
    _note_use(weight, bias)
    y = _LinearFn.apply(x2, weight, bias, r2, ACT[act], float(rscale), float(drop_p), seed)
    return y.reshape(*lead, weight.shape[0])


class _LinearCatFn(torch.autograd.Function):
    """y = [x1 | x2] @ W^T + b without materialising the concatenation
    (torch.cat([x, grid], -1) -> fc, libs/model.py:615-617).  The weight is split into two contiguous
    blocks so the wide part (K1 = n_hidden) keeps TMA-legal pitches and runs on the tensor cores; the
    2-column coordinate part is a K=2 SIMT update."""

    @staticmethod
    def forward(ctx, x1, x2, weight, bias):
        require_cuda_f32(x1, x2, weight, bias)
        M, K1 = x1.shape
        K2 = x2.shape[1]
        N, K = weight.shape
        assert K == K1 + K2
        w1 = weight[:, :K1].contiguous()
        w2 = weight[:, K1:].contiguous()
        y = torch.empty((M, N), dtype=torch.float32, device=x1.device)
        gemm(x1, w1, y, M, N, K1, lda=K1, ldb=K1, ldc=N, transB=True, bias=bias)
        gemm(x2, w2, y, M, N, K2, lda=K2, ldb=K2, ldc=N, transB=True, accumulate=True)
        ctx.save_for_backward(x1, x2, w1, w2)
        ctx.has_bias = bias is not None
        ctx.weight_ref, ctx.bias_ref = _weak(weight), _weak(bias)
        return y

    @staticmethod
    def backward(ctx, dy):
        x1, x2, w1, w2 = ctx.saved_tensors
        dy = dy.contiguous()
        M, K1 = x1.shape
        K2 = x2.shape[1]
        N = w1.shape[0]
        dx1 = dx2 = dw = db = dw1 = dw2 = None
        fork = _Fork(dy)
        if ctx.needs_input_grad[2]:
            dw1 = torch.empty_like(w1)
            dw2 = torch.empty_like(w2)
            dw = torch.empty((N, K1 + K2), dtype=torch.float32, device=dy.device)
            with fork.side(0):
                gemm(dy, x1, dw1, N, K1, M, lda=N, ldb=K1, ldc=K1, transA=True, wgrad=True)
                gemm(dy, x2, dw2, N, K2, M, lda=N, ldb=K2, ldc=K2, transA=True, wgrad=True)
                torch.cat([dw1, dw2], dim=1, out=dw)
        if ctx.has_bias and ctx.needs_input_grad[3]:
            db = torch.empty(N, dtype=torch.float32, device=dy.device)
            with fork.side(1):
                colsum(dy, M, N, N, db)
        if ctx.needs_input_grad[0]:
            dx1 = torch.empty_like(x1)
            gemm(dy, w1, dx1, M, K1, N, lda=N, ldb=K1, ldc=K1)
        if ctx.needs_input_grad[1]:
            dx2 = torch.empty_like(x2)
            gemm(dy, w2, dx2, M, K2, N, lda=N, ldb=K2, ldc=K2)
        _finish_fork(fork, (ctx.weight_ref(), ctx.bias_ref()), (dy, x1, x2, dw1, dw2))
        return dx1, dx2, dw, db


def linear_cat(x1, x2, weight, bias=None):
    lead = x1.shape[:-1]
    _note_use(weight, bias)
    y = _LinearCatFn.apply(x1.reshape(-1, x1.shape[-1]).contiguous(),
                           x2.reshape(-1, x2.shape[-1]).contiguous(), weight, bias)
    return y.reshape(*lead, weight.shape[0])


# ------------------------------------------------------------------------------------------
# Bilinear resize (align_corners=True) of channel-last grids
# ------------------------------------------------------------------------------------------
class _InterpFn(torch.autograd.Function):
    """(B, H, W, C) -> (B, Hout, Wout, C); F.interpolate(mode='bilinear', align_corners=True) of the interpolation
    scalers (libs/layers.py:431-512, 624-670) on channel-last memory; deterministic gather backward."""

    @staticmethod
    def forward(ctx, x, Hout, Wout):
        require_cuda_f32(x)
        B, H, W, C = x.shape
        y = torch.empty((B, Hout, Wout, C), dtype=torch.float32, device=x.device)
        _launch("interp_bilinear", 8.0 * y.numel(), 4.0 * (x.numel() + y.numel()), _lib.load().gb200_interp_bilinear_fwd,
                _dev(x), ptr(x), B, H, W, C, ptr(y), Hout, Wout, stream_of(x))
        ctx.shape = (B, H, W, C, Hout, Wout)
        return y

    @staticmethod
    def backward(ctx, dy):
        B, H, W, C, Hout, Wout = ctx.shape
        dy = dy.contiguous()
        dx = torch.empty((B, H, W, C), dtype=torch.float32, device=dy.device)
        _launch("interp_bilinear", 8.0 * dy.numel(), 4.0 * (dx.numel() + dy.numel()),
                _lib.load().gb200_interp_bilinear_bwd, _dev(dy), ptr(dy), B, H, W, C, ptr(dx), Hout, Wout, stream_of(dy))
        return dx, None, None


def interp_bilinear(x, Hout, Wout):
    """x: (B, H, W, C) contiguous fp32 CUDA"""
    return _InterpFn.apply(x.contiguous(), int(Hout), int(Wout))


# ------------------------------------------------------------------------------------------
# 3x3 convolution block of the interpolation scalers (csrc/conv.cu)
# ------------------------------------------------------------------------------------------
class _Conv3x3BlockFn(torch.autograd.Function):
    """y = act(dropout_p(conv3x3(x))), x (B, H, W, Cin) channel-last fp32, weight (Cout, Cin, 3, 3), stride 1, padding 1.
    Forward and input gradient: tcgen05 implicit GEMM in bf16x3 (Cin = 1: streaming stencil); weight gradient: a library
    convolution-backward call in TF32 (a contraction over all pixels, like every other weight gradient of 'x3' mode)."""

    @staticmethod
    def forward(ctx, x, weight, act, p, seed):
        require_cuda_f32(x, weight)
        lib = _lib.load()
        B, H, W, Cin = x.shape
        Cout = weight.shape[0]
        dev, st = _dev(x), stream_of(x)
        w = weight.contiguous()
        y = torch.empty((B, H, W, Cout), dtype=torch.float32, device=x.device)
        npix = B * H * W
        z = None
        if Cin == 1:
            _launch("conv1_stencil", 18.0 * npix * Cout, 4.0 * npix * (1 + Cout), lib.gb200_conv1_fwd, dev, ptr(x), ptr(w),
                    ptr(y), B, H, W, Cout, act, p, seed, st)
        else:
            CP = 64 * ((Cin + 63) // 64)
            hi = torch.empty((npix, CP), dtype=torch.bfloat16, device=x.device)
            lo = torch.empty_like(hi)
            _launch("conv_split", 4.0 * npix * Cin, 4.0 * npix * (Cin + CP), lib.gb200_conv_split, dev, ptr(x), Cin, 0, Cin,
                    npix, ptr(hi), ptr(lo), None, 0, 0, 0, 0.0, 0, None, st)
            wt = torch.empty(lib.gb200_conv3x3_pack_bytes(Cin, Cout, 0), dtype=torch.uint8, device=x.device)
            _launch("conv_pack", 0.0, 2.0 * wt.numel(), lib.gb200_conv3x3_pack, dev, ptr(w), Cin, Cout, 0, ptr(wt), st)
            if act == ACT["silu"] and (x.requires_grad or weight.requires_grad):
                z = torch.empty_like(y)
            _launch("conv3x3_tc", 18.0 * npix * Cin * Cout, 4.0 * npix * (CP + Cout) + wt.numel(), lib.gb200_conv3x3, dev,
                    ptr(hi), ptr(lo), Cin, ptr(wt), Cout, B, H, W, ptr(y), Cout, 0, ptr(z), None, 0, 0, act, p, seed, st)
        ctx.save_for_backward(x, weight, y if z is None else z)
        ctx.cfg = (act, p, seed)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, weight, yz = ctx.saved_tensors
        act, p, seed = ctx.cfg
        lib = _lib.load()
        B, H, W, Cin = x.shape
        Cout = weight.shape[0]
        dev, st = _dev(x), stream_of(x)
        dy = dy.contiguous()
        npix = B * H * W
        w = weight.contiguous()
        dx = dw = None
        if Cin == 1:
            assert act == ACT["relu"], "conv1 backward: ReLU block only"
            dw = torch.empty_like(w)
            dx = torch.empty_like(x) if ctx.needs_input_grad[0] else None
            wsb = lib.gb200_conv1_bwd_workspace_bytes(Cout)
            ws = workspace(wsb, x)
            _launch("conv1_stencil", 36.0 * npix * Cout, 8.0 * npix * Cout, lib.gb200_conv1_bwd, dev, ptr(dy), ptr(yz), ptr(x),
                    ptr(w), ptr(dx), ptr(dw), B, H, W, Cout, p, ptr(ws), wsb, st)
            return dx, dw, None, None, None
        CPo = 64 * ((Cout + 63) // 64)
        g = torch.empty((B, H, W, Cout), dtype=torch.float32, device=x.device)
        ghi = torch.empty((npix, CPo), dtype=torch.bfloat16, device=x.device)
        glo = torch.empty_like(ghi)
        _launch("conv_split", 6.0 * npix * Cout, 4.0 * npix * (3 * Cout + CPo), lib.gb200_conv_split, dev, ptr(dy), Cout, 0, Cout,
                npix, ptr(ghi), ptr(glo), ptr(yz), Cout, 0, act, p, seed, ptr(g), st)
        fork = _Fork(dy)
        if ctx.needs_input_grad[1]:
            dw = torch.empty_like(w)          # the parameter's own layout: autograd adopts it without a copy on this stream
            with fork.side(0):
                prev = torch.backends.cudnn.allow_tf32
                torch.backends.cudnn.allow_tf32 = True
                try:
                    dw.copy_(torch.ops.aten.convolution_backward(g.permute(0, 3, 1, 2), x.permute(0, 3, 1, 2), weight, None,
                                                                 [1, 1], [1, 1], [1, 1], False, [0, 0], 1,
                                                                 [False, True, False])[1])
                finally:
                    torch.backends.cudnn.allow_tf32 = prev
        if ctx.needs_input_grad[0]:
            wt = torch.empty(lib.gb200_conv3x3_pack_bytes(Cin, Cout, 1), dtype=torch.uint8, device=x.device)
            _launch("conv_pack", 0.0, 2.0 * wt.numel(), lib.gb200_conv3x3_pack, dev, ptr(w), Cin, Cout, 1, ptr(wt), st)
            dx = torch.empty_like(x)
            _launch("conv3x3_tc", 18.0 * npix * Cin * Cout, 4.0 * npix * (CPo + Cin) + wt.numel(), lib.gb200_conv3x3, dev,
                    ptr(ghi), ptr(glo), Cout, ptr(wt), Cin, B, H, W, ptr(dx), Cin, 0, None, None, 0, 0, 0, 0.0, 0, st)
        _finish_fork(fork, (weight,), (g, x))
        return dx, dw, None, None, None


def conv3x3_supported(cin, cout):
    return bool(_lib.load().gb200_conv3x3_supported(int(cin), int(cout)))


def conv3x3_block(x, weight, *, act="relu", drop_p=0.0):
    """x (B, H, W, Cin) channel-last -> act(dropout(conv3x3(x))) (B, H, W, Cout)"""
    seed = next_seed() if drop_p > 0.0 else 0
    _note_use(weight)
    return _Conv3x3BlockFn.apply(x.contiguous(), weight, ACT[act], float(drop_p), seed)


# ------------------------------------------------------------------------------------------
# Row LayerNorm
# ------------------------------------------------------------------------------------------
class _LayerNormFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, gamma, beta, eps):
        require_cuda_f32(x, gamma, beta)
        rows, width = x.shape
        y = torch.empty_like(x)
        mean = torch.empty(rows, dtype=torch.float32, device=x.device)
        rstd = torch.empty_like(mean)
        _launch("layernorm_fwd", 8.0 * rows * width, 8.0 * rows * width, _lib.load().gb200_layernorm_fwd,
                _dev(x), ptr(x), rows, width, ptr(gamma), ptr(beta), eps, ptr(y), ptr(mean), ptr(rstd),
                stream_of(x))
        ctx.save_for_backward(x, gamma, mean, rstd)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, gamma, mean, rstd = ctx.saved_tensors
        dy = dy.contiguous()
        rows, width = x.shape
        lib = _lib.load()
        dx = torch.empty_like(x)
        dg = torch.empty_like(gamma)
        db = torch.empty_like(gamma)
        ws_bytes = lib.gb200_layernorm_bwd_workspace_bytes(rows, width)
        ws = workspace(ws_bytes, x)
        _launch("layernorm_bwd", 14.0 * rows * width, 12.0 * rows * width, lib.gb200_layernorm_bwd, _dev(x),
                ptr(dy), ptr(x), ptr(mean), ptr(rstd), ptr(gamma), rows, width, ptr(dx), ptr(dg), ptr(db), 0,
                ptr(ws), ws_bytes, stream_of(x))
        return dx, dg, db, None


def layer_norm(x, gamma, beta, eps):
    shape = x.shape
    return _LayerNormFn.apply(x.reshape(-1, shape[-1]).contiguous(), gamma, beta, float(eps)).reshape(shape)


# ------------------------------------------------------------------------------------------
# Attention: Q/K/V projection + per-head LayerNorm + position columns + K^T V + Q.(.)
# ------------------------------------------------------------------------------------------
def _hop(t, ld, col0, augmented=False, gamma=None, beta=None):
    return HeadOperand(ptr(t), ld, col0, int(augmented), ptr(gamma), ptr(beta))


class _LinearAttentionFn(torch.autograd.Function):
    """(query, key, value) -> head-merged attention output (B, n, H*(p+dk)) and A (B,H,d,d).

    Galerkin  (libs/layers.py:708-734):  A = mask2 * K~^T V~ / n,           out = Q~ A
    Fourier in linear form (exact reassociation of libs/layers.py:687-703 when the n x n
    dropout is off):                     A = K~^T V~ / (sqrt(d) n),          out = Q~ A
    with ~ = [pos | per-head-LayerNorm(.)] on the operands selected by `norm_on`.
    """

    @staticmethod
    def forward(ctx, query, key, value, pos, flat, keep_mask, cfg):
        H, dk, p, eps, norm_on, scale, self_attn, mask_p, mask_seed, quadratic, want_attn = cfg
        require_cuda_f32(query, key, value, pos, flat)
        lib = _lib.load()
        B, n, dm = query.shape
        wqkv, bqkv, g1, b1, g2, b2 = _unpack_attention_params(flat, dm, H, dk, norm_on is not None)
        T, d = B * n, dk + p
        dev = _dev(query)
        st = stream_of(query)
        tc = int(_PRECISION == "tf32")
        qkv = torch.empty((T, 3 * dm), dtype=torch.float32, device=query.device)
        xs = [t.reshape(T, dm) for t in (query, key, value)]
        blocks = {"kv": (1, 2), "qk": (1, 0), None: ()}[norm_on]
        rstd = []
        if self_attn:      # one GEMM, N = 3*d_model
            gemm(xs[0], wqkv, qkv, T, 3 * dm, dm, lda=dm, ldb=dm, ldc=3 * dm, transB=True, bias=bqkv)
        else:
            for i in range(3):
                gemm(xs[i], wqkv, qkv, T, dm, dm, lda=dm, ldb=dm, ldc=3 * dm, transB=True,
                     bias=bqkv[i * dm:(i + 1) * dm], b_off=i * dm * dm, c_off=i * dm)
        # which blocks are normalised: galerkin -> (K, V), fourier -> (Q, K)
        if blocks:      # both normalised operand blocks in ONE launch
            rstd = [torch.empty((T, H), dtype=torch.float32, device=query.device) for _ in blocks]
            _launch("headnorm_fwd", 16.0 * T * dm, 16.0 * T * dm, lib.gb200_headnorm_fwd, dev, ptr(qkv), 3 * dm,
                    blocks[0] * dm, blocks[1] * dm, T, H, dk, eps, ptr(rstd[0]), ptr(rstd[1]), st)
        aff = {0: (None, None), 1: (None, None), 2: (None, None)}
        if blocks:
            aff[blocks[0]] = (g1, b1)
            aff[blocks[1]] = (g2, b2)
        ops = [_hop(qkv, 3 * dm, i * dm, False, *aff[i]) for i in range(3)]
        if quadratic:
            # (Q~ K~^T) V~ with an n x n dropout in between: flash-style quadratic kernels
            out = torch.empty((B, n, H * d), dtype=torch.float32, device=query.device)
            A = torch.empty((B, H, n, n) if want_attn else (0,), dtype=torch.float32, device=query.device)
            _launch("fourier_quad_fwd", 4.0 * B * H * n * n * d, 4.0 * (3 * T * dm + T * H * d),
                    lib.gb200_fourier_quad_fwd, dev, ops[0], ops[1], ops[2], ptr(pos), B, H, n, dk, p, scale,
                    ptr(keep_mask), mask_p, mask_seed, ptr(out), ptr(A) if want_attn else None, st)
            ctx.save_for_backward(query, key, value, pos, flat, keep_mask, qkv, A, *rstd)
            ctx.cfg = cfg
            ctx.set_materialize_grads(False)
            ctx.mark_non_differentiable(A)
            return out, A
        A = torch.empty((B, H, d, d), dtype=torch.float32, device=query.device)
        nsplit = lib.gb200_attn_suggest_nsplit(B, H, n)
        ws_bytes = lib.gb200_attn_xty_workspace_bytes(B, H, d, nsplit)
        ws = workspace(ws_bytes, qkv)
        xty_work = (2.0 * B * H * n * d * d, 4.0 * (2 * T * dm + T * p))
        xm_work = (2.0 * B * H * n * d * d, 4.0 * (T * dm + T * p + T * H * d))
        _launch("attn_xty", *xty_work, lib.gb200_attn_xty, dev, ops[1], ops[2], ptr(pos), B, H, n, dk, p, scale,
                ptr(keep_mask), mask_p, mask_seed, ptr(A), nsplit, ptr(ws), ws_bytes, tc, st)
        out = torch.empty((B, n, H * d), dtype=torch.float32, device=query.device)
        _launch("attn_xm", *xm_work, lib.gb200_attn_xm, dev, ops[0], ptr(pos), ptr(A), 0, B, H, n, dk, p,
                ptr(out), H * d, 0, 1, 1.0, tc, st)
        ctx.save_for_backward(query, key, value, pos, flat, keep_mask, qkv, A, *rstd)
        ctx.cfg = cfg
        ctx.set_materialize_grads(False)
        return out, A

    @staticmethod
    def backward(ctx, dout, dA_ext):
        (query, key, value, pos, flat, keep_mask, qkv, A, *rstd) = ctx.saved_tensors
        H, dk, p, eps, norm_on, scale, self_attn, mask_p, mask_seed, quadratic, want_attn = ctx.cfg
        lib = _lib.load()
        B, n, dm = query.shape
        wqkv, _bq, g1, b1, g2, b2 = _unpack_attention_params(flat, dm, H, dk, norm_on is not None)
        T, d = B * n, dk + p
        dev, st = _dev(query), stream_of(query)
        tc = int(_PRECISION == "tf32")
        dout = torch.zeros((B, n, H * d), dtype=torch.float32, device=query.device) if dout is None \
            else dout.contiguous()
        blocks = {"kv": (1, 2), "qk": (1, 0), None: ()}[norm_on]
        aff = {0: (None, None), 1: (None, None), 2: (None, None)}
        if blocks:
            aff[blocks[0]] = (g1, b1)
            aff[blocks[1]] = (g2, b2)
        ops = [_hop(qkv, 3 * dm, i * dm, False, *aff[i]) for i in range(3)]
        do_op = _hop(dout, H * d, 0, True)
        if quadratic:
            dqkv = torch.empty((T, 3 * dm), dtype=torch.float32, device=query.device)
            _launch("fourier_quad_bwd", 10.0 * B * H * n * n * d, 4.0 * (6 * T * dm + T * H * d),
                    lib.gb200_fourier_quad_bwd, dev, ops[0], ops[1], ops[2], do_op, ptr(pos), B, H, n, dk, p, scale,
                    ptr(keep_mask), mask_p, mask_seed, ptr(dqkv), 3 * dm, 0, dm, 2 * dm, st)
            return _LinearAttentionFn._finish_backward(ctx, dqkv, blocks, rstd, qkv, g1, g2, query, key, value, wqkv,
                                                       flat, H, dk, T, dm, self_attn, dev, st)
        # G = scale * mask2 * (Q~^T dO [+ external grad of A])
        G = torch.empty((B, H, d, d), dtype=torch.float32, device=query.device)
        xty_work = (2.0 * B * H * n * d * d, 4.0 * (T * dm + T * p + T * H * d))
        xm_work = (2.0 * B * H * n * d * d, 4.0 * (2 * T * dm + T * p))
        dqkv = torch.empty((T, 3 * dm), dtype=torch.float32, device=query.device)
        # dQ~ = dO A^T needs nothing from the G chain: side stream 0, concurrent with the contraction below
        fork = _Fork(dout)
        with fork.side(0):
            _launch("attn_xm", *xm_work, lib.gb200_attn_xm, dev, do_op, ptr(pos), ptr(A), 1, B, H, n, dk, p, ptr(dqkv),
                    3 * dm, 0, 0, 1.0, tc, stream_of(query))
        nsplit = lib.gb200_attn_suggest_nsplit(B, H, n)
        ws_bytes = lib.gb200_attn_xty_workspace_bytes(B, H, d, nsplit)
        ws = workspace(ws_bytes, qkv)
        if dA_ext is None:       # the usual case: nobody differentiates through the returned A
            _launch("attn_xty", *xty_work, lib.gb200_attn_xty, dev, ops[0], do_op, ptr(pos), B, H, n, dk, p,
                    scale, ptr(keep_mask), mask_p, mask_seed, ptr(G), nsplit, ptr(ws), ws_bytes, tc, st)
        else:
            _launch("attn_xty", *xty_work, lib.gb200_attn_xty, dev, ops[0], do_op, ptr(pos), B, H, n, dk, p, 1.0,
                    None, 0.0, 0, ptr(G), nsplit, ptr(ws), ws_bytes, tc, st)
            G = (G + dA_ext) * scale
            if keep_mask is not None:
                G = G * (2.0 * keep_mask.to(G.dtype))
            elif mask_p > 0.0:
                drop = torch.empty_like(G)
                check(lib.gb200_philox_scale(dev, ptr(drop), drop.numel(), mask_p, mask_seed, st), "gb200_philox_scale")
                G = G * drop
            G = G.contiguous()
        # dV~ = K~ G (side stream 1) ; dK~ = V~ G^T   (position columns carry no gradient)
        with fork.side(1):
            _launch("attn_xm", *xm_work, lib.gb200_attn_xm, dev, ops[1], ptr(pos), ptr(G), 0, B, H, n, dk, p, ptr(dqkv),
                    3 * dm, 2 * dm, 0, 1.0, tc, stream_of(query))
        _launch("attn_xm", *xm_work, lib.gb200_attn_xm, dev, ops[2], ptr(pos), ptr(G), 1, B, H, n, dk, p, ptr(dqkv),
                3 * dm, dm, 0, 1.0, tc, st)
        fork.join()
        return _LinearAttentionFn._finish_backward(ctx, dqkv, blocks, rstd, qkv, g1, g2, query, key, value, wqkv, flat,
                                                   H, dk, T, dm, self_attn, dev, st)

    @staticmethod
    def _finish_backward(ctx, dqkv, blocks, rstd, qkv, g1, g2, query, key, value, wqkv, flat, H, dk, T, dm, self_attn,
                         dev, st):
        """per-head LayerNorm backward on the normalised blocks, then the Q/K/V projection backward.  Every
        parameter gradient is written straight into its slice of ONE flat buffer (the gradient of the packed
        parameter vector), which _PackFn.backward hands out as views."""
        lib = _lib.load()
        dflat = torch.empty_like(flat)
        dwqkv, dbqkv, dg1, db1, dg2, db2 = _unpack_attention_params(dflat, dm, H, dk, bool(blocks))
        if blocks:
            dgb = [dg1, db1, dg2, db2]
            wsb = lib.gb200_headnorm_bwd_workspace_bytes(T, H, dk)
            w2 = workspace(wsb, qkv)
            _launch("headnorm_bwd", 28.0 * T * dm, 24.0 * T * dm, lib.gb200_headnorm_bwd, dev, ptr(dqkv), 3 * dm,
                    blocks[0] * dm, blocks[1] * dm, ptr(qkv), 3 * dm, blocks[0] * dm, blocks[1] * dm, ptr(rstd[0]),
                    ptr(rstd[1]), ptr(g1), ptr(g2), T, H, dk, ptr(dgb[0]), ptr(dgb[1]), ptr(dgb[2]), ptr(dgb[3]), 0,
                    ptr(w2), wsb, st)
        # projection backward: weight and bias gradients on side streams, input gradients on the launching one
        fork = _Fork(dqkv)
        with fork.side(1):
            colsum(dqkv, T, 3 * dm, 3 * dm, dbqkv)
        xs = [t.reshape(T, dm) for t in (query, key, value)]
        dq = dk_ = dv = None
        if self_attn:
            with fork.side(0):
                gemm(dqkv, xs[0], dwqkv, 3 * dm, dm, T, lda=3 * dm, ldb=dm, ldc=dm, transA=True, wgrad=True)
            if ctx.needs_input_grad[0]:
                dq = torch.empty_like(query)
                gemm(dqkv, wqkv, dq, T, dm, 3 * dm, lda=3 * dm, ldb=dm, ldc=dm)
        else:
            with fork.side(0):
                for i in range(3):
                    gemm(dqkv, xs[i], dwqkv, dm, dm, T, lda=3 * dm, ldb=dm, ldc=dm, transA=True, a_off=i * dm,
                         c_off=i * dm * dm, wgrad=True)
            grads = []
            for i in range(3):
                gi = None
                if ctx.needs_input_grad[i]:
                    gi = torch.empty_like(query)
                    gemm(dqkv, wqkv, gi, T, dm, dm, lda=3 * dm, ldb=dm, ldc=dm, a_off=i * dm, b_off=i * dm * dm)
                grads.append(gi)
            dq, dk_, dv = grads
        fork.join()
        return (dq, dk_, dv, None, dflat, None, None)


def _unpack_attention_params(flat, dm, H, dk, has_norm):
    """views of the packed [W_qkv (3dm,dm) | b_qkv (3dm) | gamma1 | beta1 | gamma2 | beta2 (H,dk each)] vector"""
    o = 3 * dm * dm
    wqkv = flat[:o].view(3 * dm, dm)
    bqkv = flat[o:o + 3 * dm]
    o += 3 * dm
    if not has_norm:
        return wqkv, bqkv, None, None, None, None
    tabs = [flat[o + i * dm:o + (i + 1) * dm].view(H, dk) for i in range(4)]
    return (wqkv, bqkv, *tabs)


def linear_attention(query, key, value, pos, flat, has_norm, keep_mask, *, n_head, pos_dim,
                     eps, attention_type, self_attn, mask_p=0.0, quadratic=False, want_attn=False):
    """keep_mask: explicit (B,H,d,d) uint8 keep-mask, or None with mask_p > 0 for the in-kernel Philox
    dropout of the attention matrix (no mask tensor, regenerated in backward)."""
    B, n, dm = query.shape
    dk = dm // n_head
    p = pos_dim if pos is not None else 0
    d = dk + p
    if attention_type == "galerkin":
        norm_on, scale = ("kv" if has_norm else None), 1.0 / n
    else:
        norm_on, scale = ("qk" if has_norm else None), 1.0 / (math.sqrt(d) * n)
    mask_p = 0.0 if keep_mask is not None else float(mask_p)
    cfg = (n_head, dk, p, float(eps), norm_on, float(scale), bool(self_attn), mask_p,
           next_seed() if mask_p > 0.0 else 0, bool(quadratic), bool(want_attn))
    pos_c = None if pos is None else pos.contiguous()
    return _LinearAttentionFn.apply(query.contiguous(), key.contiguous(), value.contiguous(), pos_c, flat, keep_mask,
                                    cfg)


# ------------------------------------------------------------------------------------------
# Fused encoder layer (csrc/encoder_fwd.cu): three tcgen05 kernels per layer forward
# ------------------------------------------------------------------------------------------
# The launching stream joins the weight-gradient side stream only when the whole backward pass is enqueued (autograd engine
# callback), so the grouped weight-gradient GEMM of layer l overlaps the input-gradient chain of layers l-1, l-2, ...
# Measured at C3 with the grouped launch: 4.82 -> 4.67 ms/step.  Joining per layer instead is what graphs.GraphedStep
# selects for concurrent micro-batch chains, whose per-chain streams are joined before the backward pass ends
# (_DEFER_WGRAD_JOIN is defined next to _Fork)


class _Ctx:
    """stand-in autograd context for calling another Function's backward on explicit tensors"""

    def __init__(self, saved, cfg, needs):
        self.saved_tensors, self.cfg, self.needs_input_grad = saved, cfg, needs


def encoder_pack(params, H, dm, p, dff):
    """parameters -> bf16 (hi, lo) operand tile streams + fp32 vector block of the fused kernels (one launch)"""
    lib = _lib.load()
    P, _ = _encoder_params_struct(params, H, dm, p, dff)
    packed = torch.empty(lib.gb200_encoder_pack_bytes(dm, H, p, dff), dtype=torch.uint8, device=params[0].device)
    _launch("encoder_pack", 0.0, 2.0 * packed.numel(), lib.gb200_encoder_pack, _dev(packed), ctypes.byref(P), ptr(packed),
            stream_of(packed))
    return packed


def encoder_fused_supported(d_model, n_head, pos_dim, d_ff):
    return bool(_lib.load().gb200_encoder_supported(int(d_model), int(n_head), int(pos_dim), int(d_ff)))


def _encoder_params_struct(params, H, dm, p, dff):
    (wq, wk, wv, bq, bk, bv, *rest) = params
    P = _lib.EncoderParams()
    P.wq, P.wk, P.wv, P.bq, P.bk, P.bv = (ptr(t) for t in (wq, wk, wv, bq, bk, bv))
    has_norm = len(rest) == 4 * H + 6
    if has_norm:
        for h in range(H):
            P.gamma_k[h], P.beta_k[h] = ptr(rest[h]), ptr(rest[H + h])
            P.gamma_v[h], P.beta_v[h] = ptr(rest[2 * H + h]), ptr(rest[3 * H + h])
        rest = rest[4 * H:]
    P.wfc, P.bfc, P.w1, P.b1, P.w2, P.b2 = (ptr(t) for t in rest)
    P.d_model, P.n_head, P.pos_dim, P.d_ff = dm, H, p, dff
    return P, has_norm


class _EncoderLayerFn(torch.autograd.Function):
    """One Galerkin encoder layer (libs/model.py:104-140) as ONE autograd node.

    params = (Wq, Wk, Wv, bq, bk, bv, [gamma_K x H, beta_K x H, gamma_V x H, beta_V x H,] W_fc, b_fc, W1, b1, W2, b2)
    forward : gb200_encoder_pack + gb200_encoder_layer_fwd (3 kernels)
    backward: the per-operator backward launches on the tensors the fused forward saved (same layouts, same Philox
              streams), see _LinearAttentionFn / _LinearFn / _MLP2Fn."""

    @staticmethod
    def forward(ctx, x, pos, keep_mask, cfg, packed, *params):
        (H, p, eps, scale, mask_p, mask_seed, p1, seed1, sign, pf, seedf, p2, seed2) = cfg
        require_cuda_f32(x, pos, *params)
        lib = _lib.load()
        B, n, dm = x.shape
        dk, d = dm // H, dm // H + p
        dff = params[-4].shape[0]
        T = B * n
        dev, st = _dev(x), stream_of(x)
        has_norm = len(params) == 4 * H + 12
        if packed is None:
            packed = encoder_pack(params, H, dm, p, dff)
        f32 = dict(dtype=torch.float32, device=x.device)
        qkv = torch.empty((T, 3 * dm), **f32)
        rstd = [torch.empty((T, H), **f32) for _ in range(2)] if has_norm else [None, None]
        A = torch.empty((B, H, d, d), **f32)
        heads = torch.empty((B, n, H * d), **f32)
        x1 = torch.empty((T, dm), **f32)
        hid = torch.empty((T, dff), **f32)
        x2 = torch.empty((B, n, dm), **f32)
        wsb = lib.gb200_encoder_workspace_bytes(B, n, H, dk, p)
        ws = workspace(wsb, x)
        # ALGORITHMIC work per kernel (DESIGN.md section 3): flops of the GEMMs it carries, bytes of the tensors it must read / write
        work = {1: ("enc_qkv", 2.0 * T * 3 * dm * dm + 2.0 * B * H * n * d * d, 4.0 * T * (dm + 3 * dm + 2 * H) + 2.0 * 3 * dm * dm),
                2: ("enc_attn", 2.0 * B * H * n * d * d + 2.0 * T * H * d * dm, 4.0 * T * (dm + H * d + 2 * dm) + 2.0 * H * d * dm),
                4: ("enc_ffn", 4.0 * T * dm * dff, 4.0 * T * (dm + dff + dm) + 4.0 * dm * dff)}
        args = (dev, ptr(packed), dm, H, p, dff, ptr(x), ptr(pos), B, n, int(has_norm), eps, scale, ptr(keep_mask), mask_p,
                mask_seed, p1, seed1, sign, pf, seedf, p2, seed2, ptr(qkv), ptr(rstd[0]), ptr(rstd[1]), ptr(A), ptr(heads),
                ptr(x1), ptr(hid), ptr(x2), ptr(ws), wsb)
        if Profiler.enabled:       # attribution pass: one launch per event pair
            for bit, (fam, fl, by) in work.items():
                _launch(fam, fl, by, lib.gb200_encoder_layer_fwd, *args, bit, st)
        else:
            _launch("encoder_layer_fwd", sum(w[1] for w in work.values()), sum(w[2] for w in work.values()),
                    lib.gb200_encoder_layer_fwd, *args, 7, st)
        ctx.save_for_backward(x, pos, keep_mask, qkv, A, heads, x1, hid, packed, *[r for r in rstd if r is not None],
                              *params)
        ctx.cfg = cfg
        ctx.has_norm = has_norm
        ctx.set_materialize_grads(False)
        return x2, A

    @staticmethod
    def backward(ctx, dy, dA_ext):
        (x, pos, keep_mask, qkv, A, heads, x1, hid, packed, *rest) = ctx.saved_tensors
        (H, p, eps, scale, mask_p, mask_seed, p1, seed1, sign, pf, seedf, p2, seed2) = ctx.cfg
        has_norm = ctx.has_norm
        rstd = rest[:2] if has_norm else []
        params = rest[2:] if has_norm else rest
        B, n, dm = x.shape
        dk = dm // H
        T = B * n
        wfc, bfc, w1, b1, w2, b2 = params[-6:]
        if dy is None:
            dy = torch.zeros_like(x)
        dy2 = dy.reshape(T, dm).contiguous()
        if dA_ext is None:       # the per-operator backward below also differentiates through the returned attention matrix
            return _EncoderLayerFn._backward_fused(ctx, dy2, x, pos, keep_mask, qkv, A, heads, x1, hid, packed, rstd, params)
        # FeedForward + shortcut
        c = _Ctx((x1, w1, w2, hid, None), (ACT["relu"], pf, seedf, p2, seed2, 1.0, True, True, True), (True,) * 12)
        dx1, dw1, db1, dw2, db2 = _MLP2Fn.backward(c, dy2)[:5]
        # fc + residual
        c = _Ctx((heads.reshape(T, -1), wfc, None, None), (0, sign, p1, seed1, True, True), (True,) * 8)
        dheads, dwfc, dbfc, dres = _LinearFn.backward(c, dx1)[:4]
        # attention core + per-head LayerNorm + Q/K/V projection
        flat = pack([t for t in params[:6]] + [t for t in params[6:-6]]).detach()
        acfg = (H, dk, p, eps, "kv" if has_norm else None, scale, True, mask_p, mask_seed, False, False)
        c = _Ctx((x, x, x, pos, flat, keep_mask, qkv, A, *rstd), acfg, (ctx.needs_input_grad[0],) + (False,) * 6)
        dq, _, _, _, dflat, _, _ = _LinearAttentionFn.backward(c, dheads.view(B, n, -1), dA_ext)
        dx = None
        if ctx.needs_input_grad[0]:
            dx = dq + dres.view(B, n, dm)
        o = 3 * dm * dm
        grads = [dflat[i * dm * dm:(i + 1) * dm * dm].view(dm, dm) for i in range(3)]
        grads += [dflat[o + i * dm:o + (i + 1) * dm] for i in range(3)]
        o += 3 * dm
        if has_norm:
            grads += [dflat[o + i * dk:o + (i + 1) * dk] for i in range(4 * H)]
        grads += [dwfc, dbfc, dw1, db1, dw2, db2]
        return (dx, None, None, None, None, *grads)


    @staticmethod
    def _backward_fused(ctx, dy2, x, pos, keep_mask, qkv, A, heads, x1, hid, packed, rstd, params):
        """csrc/encoder_bwd.cu: four fused kernels on the launching stream; the four weight-gradient GEMMs (TF32 tcgen05,
        contractions over all tokens) fork onto the side streams as soon as their operands exist."""
        (H, p, eps, scale, mask_p, mask_seed, p1, seed1, sign, pf, seedf, p2, seed2) = ctx.cfg
        lib = _lib.load()
        B, n, dm = x.shape
        dk, d = dm // H, dm // H + p
        dff = hid.shape[1]
        T = B * n
        dev, st = _dev(x), stream_of(x)
        has_norm = ctx.has_norm
        f32 = dict(dtype=torch.float32, device=x.device)
        g2 = torch.empty((T, dm), **f32) if p2 > 0.0 else None
        need_gfc = p1 > 0.0 or sign != 1.0
        gfc = torch.empty((T, dm), **f32) if need_gfc else None
        g1 = torch.empty((T, dff), **f32)
        dx1 = torch.empty((T, dm), **f32)
        dqkv = torch.empty((T, 3 * dm), **f32)
        dx = torch.empty((B, n, dm), **f32)
        dvec = torch.empty(3 * dm + 4 * dm + dm + dff + dm, **f32)
        # every weight gradient is its own tensor: autograd then adopts it as .grad without a copy kernel (a view, or a tensor
        # somebody else still references, would be cloned on the launching stream before the side-stream GEMM has written it)
        dw2, dw1, dwfc = torch.empty_like(params[-2]), torch.empty_like(params[-4]), torch.empty_like(params[-6])
        dwq, dwk, dwv = (torch.empty((dm, dm), **f32) for _ in range(3))
        wsb = lib.gb200_encoder_bwd_workspace_bytes(B, n, H, dk, p)
        ws = workspace(wsb, x)

        names = {1: "enc_ffn_bwd", 2: "enc_attn_bwd", 4: "enc_kv_bwd", 8: "enc_dx", 16: "enc_reduce"}

        def stage(bits, flops, nbytes):
            _launch(names[bits], flops, nbytes, lib.gb200_encoder_layer_bwd, dev, ptr(packed), dm, H, p, dff, ptr(dy2),
                    ptr(pos), B, n, int(has_norm), scale, ptr(keep_mask), mask_p, mask_seed, p1, seed1, sign, pf, p2, seed2,
                    ptr(qkv), ptr(rstd[0]) if has_norm else None, ptr(rstd[1]) if has_norm else None, ptr(A), ptr(hid),
                    ptr(g2), ptr(g1), ptr(dx1), ptr(gfc), ptr(dqkv), ptr(dx), ptr(dvec), ptr(ws), wsb, bits, st)

        fork = _Fork(dy2)
        stage(1, 4.0 * T * dm * dff, 4.0 * T * (dm + dff + dff + dm) + 4.0 * dm * dff)                 # dy, hid -> g1, dx1
        stage(2, 2.0 * T * H * d * dm + 4.0 * B * H * n * d * d, 4.0 * T * (dm + dm + dm) + 2.0 * H * d * dm)    # dx1, Q -> dQ (+G)
        stage(4, 4.0 * B * H * n * d * d, 4.0 * T * (2 * dm + 2 * dm + 2 * H))                         # x^K, x^V -> dK, dV
        stage(8, 2.0 * T * 3 * dm * dm, 4.0 * T * (3 * dm + dm + dm) + 2.0 * 3 * dm * dm)              # dqkv, dx1 -> dx
        with fork.side(0):      # the four weight gradients of the layer: one grouped split-K launch + one reduction
            x2d = x.reshape(T, dm)
            wgrad_group([(g2 if g2 is not None else dy2, dm, dm, hid, dff, dw2),
                         (g1, dff, dff, x1, dm, dw1),
                         (gfc if gfc is not None else dx1, dm, dm, heads.reshape(T, H * d), H * d, dwfc),
                         (dqkv, dm, 3 * dm, x2d, dm, dwq), (dqkv[:, dm:], dm, 3 * dm, x2d, dm, dwk),
                         (dqkv[:, 2 * dm:], dm, 3 * dm, x2d, dm, dwv)], T)
        stage(16, 0.0, 0.0)
        _finish_fork(fork, params, (dy2, g2, g1, dx1, gfc, dqkv, hid, x1, heads, x))
        grads = [dwq, dwk, dwv] + [dvec[i * dm:(i + 1) * dm] for i in range(3)]
        o = 3 * dm
        if has_norm:
            grads += [dvec[o + i * dk:o + (i + 1) * dk] for i in range(4 * H)]
        o += 4 * dm
        grads += [dwfc, dvec[o:o + dm], dw1, dvec[o + dm:o + dm + dff], dw2, dvec[o + dm + dff:o + 2 * dm + dff]]
        return (dx if ctx.needs_input_grad[0] else None, None, None, None, None, *grads)


def encoder_layer(x, pos, params, *, n_head, pos_dim, eps, attention_scale, keep_mask=None, mask_p=0.0,
                  p_attn_out=0.0, res_sign=1.0, p_ffn=0.0, p_out=0.0, packed=None):
    """Fused Galerkin encoder layer; returns (x_out (B, n, d_model), attention matrix (B, H, d, d))."""
    mask_p = 0.0 if keep_mask is not None else float(mask_p)
    cfg = (int(n_head), int(pos_dim), float(eps), float(attention_scale), mask_p,
           next_seed() if mask_p > 0.0 else 0, float(p_attn_out), next_seed() if p_attn_out > 0.0 else 0,
           float(res_sign), float(p_ffn), next_seed() if p_ffn > 0.0 else 0, float(p_out),
           next_seed() if p_out > 0.0 else 0)
    _note_use(*params)
    return _EncoderLayerFn.apply(x.contiguous(), pos.contiguous(), keep_mask, cfg, packed, *params)


# ------------------------------------------------------------------------------------------
# Spectral convolution
# ------------------------------------------------------------------------------------------
_twiddle_cache = {}


def _twiddles(n, m, device, two_d):
    """(cos, sin)(2 pi k j / n) tables, computed in float64 once per (n, m, device)."""
    key = (n, m, str(device), two_d)
    tw = _twiddle_cache.get(key)
    if tw is None:
        j = torch.arange(n, dtype=torch.float64)
        ky = torch.arange(m, dtype=torch.float64)
        th = 2.0 * math.pi * torch.outer(ky, j) / n
        twY = torch.stack([th.cos(), th.sin()], -1).to(torch.float32).to(device).contiguous()
        twX = None
        if two_d:
            r = torch.arange(2 * m)
            kx = torch.where(r < m, r, n - 2 * m + r).to(torch.float64)
            ps = 2.0 * math.pi * torch.outer(kx, j) / n
            twX = torch.stack([ps.cos(), ps.sin()], -1).to(torch.float32).to(device).contiguous()
        tw = (twY, twX)
        _twiddle_cache[key] = tw
    return tw


def _ydft(x, R, n, C, m, twY, scale, hermitian):
    lib = _lib.load()
    out = torch.empty((R, m, C, 2), dtype=torch.float32, device=x.device)
    nsplit = lib.gb200_spectral_suggest_ysplit(R, C, n)
    ws_bytes = lib.gb200_spectral_ydft_workspace_bytes(R, C, m, nsplit)
    ws = workspace(ws_bytes, x)
    _launch("spectral_ydft", 4.0 * R * n * C * m, 4.0 * R * n * C + 8.0 * R * m * C, lib.gb200_spectral_ydft,
            _dev(x), ptr(x), R, n, C, m, ptr(twY), scale, int(hermitian), ptr(out), nsplit, ptr(ws), ws_bytes,
            int(_PRECISION == "tf32"), stream_of(x))
    return out


def _xdft(t, B, n, m, C, twX, scale, inverse):
    lib = _lib.load()
    shape = (B, n, m, C, 2) if inverse else (B, 2 * m, m, C, 2)
    out = torch.empty(shape, dtype=torch.float32, device=t.device)
    _launch("spectral_xdft", 16.0 * B * n * m * m * C, 8.0 * B * (n + 2 * m) * m * C, lib.gb200_spectral_xdft,
            _dev(t), ptr(t), B, n, m, C, ptr(twX), scale, int(inverse), ptr(out), stream_of(t))
    return out


def _yidft_epi(Z, R, n, m, Co, twY, scale, hermitian, x2, Ci, Wm, bias, act, want_z):
    lib = _lib.load()
    y = torch.empty((R, n, Co), dtype=torch.float32, device=Z.device)
    z = torch.empty_like(y) if want_z else None
    _launch("spectral_yidft_epilogue", R * n * Co * (4.0 * m + 2.0 * Ci),
            4.0 * R * n * (Ci + Co * (1 + want_z)) + 8.0 * R * m * Co + 4.0 * Ci * Co,
            lib.gb200_spectral_yidft_epilogue, _dev(Z), ptr(Z), R, n, m, Co, ptr(twY), scale, int(hermitian),
            ptr(x2), Ci, ptr(Wm), ptr(bias), act, ptr(y), ptr(z), int(_PRECISION == "tf32"), stream_of(Z))
    return y, z


class _SpectralConvFn(torch.autograd.Function):
    """act( irfft( W . rfft(x)[modes] ) + x @ Wl^T + bl ), channel-last, 1-D or 2-D
    (libs/layers.py:1077-1106 and :1153-1197).  Optionally also returns the kept-mode block of
    out_ft (B, halves*M2, Co, 2) for the `return_freq` contract."""

    @staticmethod
    def forward(ctx, x, xf, wl, bl, fw0, fw1, modes, act, two_d):
        # x feeds the pointwise residual path, xf the transform (xf is x unless the module's
        # input dropout is active: libs/layers.py:1083-1084, 1172-1173)
        require_cuda_f32(x, xf, wl, bl, fw0, fw1)
        same = xf is None
        xf = x if same else xf
        lib = _lib.load()
        m = modes
        if two_d:
            B, n, n2, Ci = x.shape
            assert n == n2
        else:
            B, n, Ci = x.shape
        Co = wl.shape[0]
        if 2 * m > n and two_d:
            raise NotImplementedError(f"SpectralConv2d: 2*modes={2*m} > n={n} (overlapping mode blocks)")
        if m > n // 2 + 1:
            raise NotImplementedError(f"SpectralConv: modes={m} > n//2+1 for n={n}")
        twY, twX = _twiddles(n, m, x.device, two_d)
        dev, st = _dev(x), stream_of(x)
        halves, M2 = (2, m * m) if two_d else (1, m)
        if two_d:
            T1 = _ydft(xf, B * n, n, Ci, m, twY, 1.0, False)
            Xf = _xdft(T1, B, n, m, Ci, twX, 1.0 / n, False)
        else:
            Xf = _ydft(xf, B, n, Ci, m, twY, 1.0 / math.sqrt(n), False)
        Of = torch.empty((B, halves * M2, Co, 2), dtype=torch.float32, device=x.device)
        mix_work = (8.0 * B * halves * M2 * Ci * Co, 8.0 * halves * M2 * (Ci * Co + B * (Ci + Co)))
        _launch("spectral_mix", *mix_work, lib.gb200_spectral_mix_fwd, dev, ptr(Xf), ptr(fw0), ptr(fw1), B, halves,
                M2, Ci, Co, ptr(Of), st)
        wm = wl.t().contiguous()                      # (Ci, Co): coalesced over output channels
        need_z = act != 0 and (x.requires_grad or wl.requires_grad or fw0.requires_grad)
        if two_d:
            Z = _xdft(Of, B, n, m, Co, twX, 1.0, True)
            y, z = _yidft_epi(Z, B * n, n, m, Co, twY, 1.0 / n, True, x, Ci, wm, bl, act, need_z)
            y = y.view(B, n, n, Co)
        else:
            y, z = _yidft_epi(Of, B, n, m, Co, twY, 1.0 / math.sqrt(n), True, x, Ci, wm, bl, act, need_z)
        ctx.save_for_backward(x, wl, fw0, fw1, Xf, z)
        ctx.cfg = (m, act, two_d, bl is not None, same)
        ctx.bias_ref = _weak(bl)
        ctx.mark_non_differentiable(Of)
        return y, Of

    @staticmethod
    def backward(ctx, gy, _gof):
        x, wl, fw0, fw1, Xf, z = ctx.saved_tensors
        m, act, two_d, has_bias, same = ctx.cfg
        lib = _lib.load()
        if two_d:
            B, n, _, Ci = x.shape
        else:
            B, n, Ci = x.shape
        Co = wl.shape[0]
        P = B * n * n if two_d else B * n
        twY, twX = _twiddles(n, m, x.device, two_d)
        dev, st = _dev(x), stream_of(x)
        halves, M2 = (2, m * m) if two_d else (1, m)
        gy = gy.contiguous()
        dbl = None
        if act != 0 and has_bias and ctx.needs_input_grad[3]:
            gz = torch.empty((P, Co), dtype=torch.float32, device=x.device)
            dbl = torch.empty(Co, dtype=torch.float32, device=x.device)
            wsb = lib.gb200_epilogue_bwd_bias_workspace_bytes(P, Co)
            wsp = workspace(wsb, x)
            _launch("epilogue_bwd_bias", 5.0 * P * Co, 12.0 * P * Co, lib.gb200_epilogue_bwd_bias, dev, ptr(gy), Co,
                    ptr(z), Co, None, Co, ptr(gz), Co, P, Co, act, 1.0, 0.0, 0, ptr(dbl), ptr(wsp), wsb, st)
        else:
            gz = epilogue_bwd(gy, P, Co, z=z, act=act) if act != 0 else gy
        # parameter gradients leave the critical path (side streams, joined at the end of this node): the pointwise weight
        # needs only gz, the spectral weights only dO^
        fork = _Fork(gz)
        dwl = None
        if ctx.needs_input_grad[2]:
            dwl = torch.empty_like(wl)
            with fork.side(0):
                gemm(gz, x, dwl, Co, Ci, P, lda=Co, ldb=Ci, ldc=Ci, transA=True, wgrad=True)
        if dbl is None and has_bias and ctx.needs_input_grad[3]:
            dbl = torch.empty(Co, dtype=torch.float32, device=x.device)
            with fork.side(0):
                colsum(gz, P, Co, Co, dbl)
        # adjoint of the inverse transform:  dO^ = (c_ky s) * DFT(gz) on the kept modes
        if two_d:
            dZ = _ydft(gz, B * n, n, Co, m, twY, 1.0 / n, True)
            dO = _xdft(dZ, B, n, m, Co, twX, 1.0, False)
        else:
            dO = _ydft(gz, B, n, Co, m, twY, 1.0 / math.sqrt(n), True)
        need_dx = ctx.needs_input_grad[0] or ctx.needs_input_grad[1]
        dXf = torch.empty((B, halves * M2, Ci, 2), dtype=torch.float32, device=x.device) if need_dx else None
        dfw0 = torch.empty_like(fw0) if ctx.needs_input_grad[4] else None
        dfw1 = torch.empty_like(fw1) if (fw1 is not None and dfw0 is not None) else None
        mix_work = (16.0 * B * halves * M2 * Ci * Co, 8.0 * halves * M2 * (2 * Ci * Co + 2 * B * (Ci + Co)))
        if dfw0 is not None:
            with fork.side(1):
                _launch("spectral_mix", mix_work[0] / 2, mix_work[1] / 2, lib.gb200_spectral_mix_bwd, dev, ptr(Xf), ptr(dO),
                        ptr(fw0), ptr(fw1), B, halves, M2, Ci, Co, None, ptr(dfw0), ptr(dfw1), 0, stream_of(dO))
        if dXf is not None:
            _launch("spectral_mix", mix_work[0] / 2, mix_work[1] / 2, lib.gb200_spectral_mix_bwd, dev, ptr(Xf), ptr(dO),
                    ptr(fw0), ptr(fw1), B, halves, M2, Ci, Co, ptr(dXf), None, None, 0, st)
        dx = dxf = None
        if need_dx:
            # adjoint of the forward transform + the pointwise path  gz @ Wl, one fused kernel
            wres = wl if same else torch.zeros_like(wl)
            if two_d:
                dT1 = _xdft(dXf, B, n, m, Ci, twX, 1.0 / n, True)
                dx, _ = _yidft_epi(dT1, B * n, n, m, Ci, twY, 1.0, False, gz, Co, wres, None, 0, False)
            else:
                dx, _ = _yidft_epi(dXf, B, n, m, Ci, twY, 1.0 / math.sqrt(n), False, gz, Co, wres, None, 0, False)
            dx = dx.view(x.shape)
            if not same:
                dxf = dx
                dx = torch.empty_like(x)
                gemm(gz, wl, dx, P, Ci, Co, lda=Co, ldb=Ci, ldc=Ci)
        _finish_fork(fork, (wl, fw0, fw1, ctx.bias_ref()), (gz, x, Xf, dO))
        return dx, dxf, dwl, dbl, dfw0, dfw1, None, None, None


def spectral_conv(x, wl, bl, fw0, fw1, *, modes, act, two_d, x_transform=None):
    """x_transform: the (dropped-out) tensor fed to the transform when it differs from x."""
    xf = None if x_transform is None else x_transform.contiguous()
    _note_use(wl, bl, fw0, fw1)
    return _SpectralConvFn.apply(x.contiguous(), xf, wl, bl, fw0, fw1, int(modes), ACT[act], bool(two_d))
