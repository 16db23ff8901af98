"""torch.autograd.Function wrappers over the C ABI (include/deer_b200.h).

PyTorch is plumbing here: it owns device memory, streams and the autograd tape; every floating-point
operation on the path runs in a hand-written sm_100a kernel of libdeer_b200.so.  All functions require
fp32 CUDA tensors and raise otherwise (no CPU / eager fallback).
"""
from __future__ import annotations

from typing import List, Optional, Sequence

import torch

from . import _lib
from ._lib import call, ptr

ACT = {"none": 0, None: 0, "relu": 1, "tanh": 2, "sigmoid": 3}
ENGINE_AUTO, ENGINE_SIMT, ENGINE_TF32, ENGINE_X3 = 0, 1, 2, 5

# Precision policy (DESIGN.md "numerics"): the time-batched contractions (M = B*T rows: LSTM input projections,
# pooling scorers, Conv1d taps) and every backward GEMM run on the tcgen05 TF32 engine; the FORWARD of the small
# post-pooling layers (M = B rows; ~25 chained GEMMs through fusion and the NIG head, <1% of the FLOPs) stays on the
# exact-fp32 engine, because TF32 rounding compounding through that chain is what pushes the NIG parameters past the
# 1e-3 relative tolerance.  The same layers' backward GEMMs are also kept exact by default: their (cancellation-
# prone) outputs feed the bias / scorer gradients whose per-tensor cosine otherwise sits at 0.9992, too close to the
# 0.999 gate (tools/precision_probe.py).
_state = {"engine": ENGINE_AUTO, "lstm_engine": ENGINE_AUTO, "exact_small_fwd": True, "exact_small_bwd": True,
          "small_rows": 8192, "direct_grad": False, "lstm_gemm16": True, "fuse_lstm_dropout": True,
          "branch_streams": True, "lstm_pre16": True, "defer_wgrad": True,
          "branch_max_batch": 512, "scorer_pool_fused": True, "grouped_batched": True, "exact_engine": ENGINE_X3,
          "small_rows_bwd": 8192, "conv_exact": 0, "lstm_keep16": True,
          "split_fwd": True, "split_rows": 1024, "bwd16": False}


def set_backward_bf16(on: bool):
    """Ablation switch (default OFF): time-batched BACKWARD contractions (>= small_rows_bwd rows) on the 16-bit tcgen05
    engine with BF16 operands instead of the TF32 engine.  Gradients tolerate the operand precision (all parity gates
    hold) and the GEMMs themselves run ~2.5x faster, but the fp32 -> BF16 cast passes of dy / x / W that feed them cost
    more than that saves: measured 4.28 ms vs 4.20 ms per B=256 step.  It would need the casts fused into the producing
    kernels (BatchNorm / scorer backward) to pay."""
    _state["bwd16"] = bool(on)


def _bwd16_ok(M: int) -> bool:
    return (_state["bwd16"] and _state["engine"] == ENGINE_AUTO and _state["lstm_gemm16"] and
            M >= _state["small_rows_bwd"] and M > 128)


def set_lstm_keep16(on: bool):
    """FP16 (default) or fp32 kept gates / cell states of the persistent LSTM kernels (DEER_OPT_LSTM_KEEP16).  Must not
    change between a forward and its backward."""
    _state["lstm_keep16"] = bool(on)
    _lib.set_option(11, 1 if on else 0)


def set_grouped_batched(on: bool):
    """Per-head grouped Linear layers as one batched GEMM launch when their operands are evenly spaced (default)."""
    _state["grouped_batched"] = bool(on)


def set_defer_wgrad(on: bool):
    """Trainer mode: weight gradients of the small (M = batch rows) Linear layers on a second stream (default on)."""
    _state["defer_wgrad"] = bool(on)


_wgrad = {"streams": {}, "pending": False}


def _wgrad_stream():
    dev = torch.cuda.current_device()
    st = _wgrad["streams"]
    if dev not in st:
        st[dev] = torch.cuda.Stream(device=dev)
    return st[dev]


def join_wgrad_stream():
    """Make the current stream wait for the deferred weight-gradient GEMMs (call after backward, before the grads are
    read).  A no-op when nothing was deferred."""
    if _wgrad["pending"]:
        torch.cuda.current_stream().wait_stream(_wgrad_stream())
        _wgrad["pending"] = False


_timeline = {"buf": None, "names": []}


def timeline_begin(device) -> None:
    """Debug aid (tools/step_timeline.py): from now on `mark(name)` launches a timestamp kernel on the current stream."""
    _timeline["buf"] = torch.zeros(256, dtype=torch.int64, device=device)
    _timeline["names"] = []


def timeline_end():
    """-> [(name, ns)] of the marks reached by the last run (after a synchronize), and stop marking."""
    buf, names = _timeline["buf"], _timeline["names"]
    _timeline["buf"] = None
    if buf is None:
        return []
    vals = buf.cpu().tolist()
    return [(n, vals[i]) for i, n in enumerate(names)]


def timeline_read():
    buf, names = _timeline["buf"], _timeline["names"]
    vals = buf.cpu().tolist()
    return [(n, vals[i]) for i, n in enumerate(names)]


def mark(name: str) -> None:
    """No-op unless a timeline is being recorded."""
    buf = _timeline["buf"]
    if buf is None:
        return
    names = _timeline["names"]
    if name in names:
        idx = names.index(name)
    else:
        idx = len(names)
        names.append(name)
    call("deer_timestamp", buf.data_ptr(), idx)


class _Mark(torch.autograd.Function):
    """Identity whose forward and backward each drop a timeline mark on their stream."""

    @staticmethod
    def forward(ctx, x, name):
        ctx.name = name
        mark(name + ":fwd")
        return x.view_as(x)

    @staticmethod
    def backward(ctx, g):
        mark(ctx.name + ":bwd")
        return g, None


def mark_tensor(x, name: str):
    return _Mark.apply(x, name) if _timeline["buf"] is not None else x


def set_lstm_pre16(on: bool):
    """FP16 (default) or fp32 pre-activations between the LSTM input projection and the recurrence kernel."""
    _state["lstm_pre16"] = bool(on)


def set_branch_streams(on: bool):
    """Run the video and text encoders of the sequence model on a second CUDA stream beside the audio LSTM (default)."""
    _state["branch_streams"] = bool(on)


def branch_streams_enabled() -> bool:
    return _state["branch_streams"]


def branch_max_batch() -> int:
    return _state["branch_max_batch"]


def set_text_stream(on: bool):
    """Text encoder on a third stream beside the video encoder (when the encoders are forked at all); off: video and
    text share the calling stream (the round-1 schedule)."""
    _state["text_stream"] = bool(on)


def text_stream_enabled() -> bool:
    return _state.get("text_stream", True)


def set_branch_max_batch(n: int):
    """Largest batch for which the sequence model forks its encoders onto two streams (default 512)."""
    _state["branch_max_batch"] = int(n)


def set_fuse_lstm_dropout(on: bool):
    """Inter-layer LSTM dropout fused into the next layer's 16-bit operand casts (default) or run as its own kernel."""
    _state["fuse_lstm_dropout"] = bool(on)


def set_lstm_gemm16(on: bool):
    """Route the LSTM layer's time-batched GEMMs through the 16-bit tcgen05 engine (default) or the TF32 engine."""
    _state["lstm_gemm16"] = bool(on)


def set_direct_grad_accumulation(on: bool):
    """Trainer mode: parameter gradients are ACCUMULATED by the backward kernels straight into the pre-allocated
    `param.grad` (views of the trainer's flat gradient buffer, zeroed once per step) and the autograd functions
    return None for them - no per-parameter temporary, zero-fill or `grad += new` launch."""
    _state["direct_grad"] = bool(on)


def _acc(param, like=None):
    """(buffer the kernels accumulate d/dparam into, whether it is param.grad itself)."""
    if param is None:
        return None, False
    if _state["direct_grad"]:
        if param.is_leaf:
            g = param.grad
            if g is not None and g.is_contiguous() and g.dtype == torch.float32 and g.is_cuda:
                return g, True
        else:
            # a view of a leaf parameter (the V rows of a packed in_proj_weight): accumulate into the same view of the
            # leaf's gradient -- no temporary, no zero fill, no slice-backward copy + add
            base = param._base
            if (base is not None and base.is_leaf and base.grad is not None and base.grad.is_contiguous() and
                    base.is_contiguous() and base.grad.dtype == torch.float32 and param.is_contiguous()):
                gv = base.grad.as_strided(param.shape, param.stride(),
                                          base.grad.storage_offset() + param.storage_offset() - base.storage_offset())
                return gv, True
    return torch.zeros_like(param if like is None else like), False


# ------------------------------------------------------------------------------------------------ zeroed scratch arena
# Transient zero-initialised scratch of the backward kernels (split-K / atomically accumulated gradient staging, the loss
# statistics): sub-allocated from one buffer that is cleared ONCE per step by one deer_fill_zero launch (begin_step)
# instead of one at::fill kernel per request.  Invariant: [cursor, zeroed) is clean.  Buffers are never freed while the
# process lives: captured CUDA graphs hold their addresses.
_arena = {}


def _arena_state(device):
    key = device.index if device.index is not None else torch.cuda.current_device()
    st = _arena.get(key)
    if st is None:
        st = _arena[key] = {"buf": None, "cursor": 0, "high": 0, "zeroed": 0, "old": []}
    return st


def _arena_begin_step():
    for st in _arena.values():
        if st["buf"] is not None and st["high"] > 0 and st["buf"].device.index == torch.cuda.current_device():
            call("deer_fill_zero", ptr(st["buf"]), st["high"], None, 0)
            st["zeroed"] = st["high"]
        st["cursor"] = 0


def zeros_scratch(shape, device) -> torch.Tensor:
    """Zero-filled fp32 scratch valid until the end of the calling autograd function (see _arena above)."""
    if isinstance(shape, int):
        shape = (shape,)
    n = 1
    for d in shape:
        n *= int(d)
    npad = (n + 63) // 64 * 64            # 256-byte slots
    st = _arena_state(torch.device(device))
    if st["cursor"] > (1 << 26) and not torch.cuda.is_current_stream_capturing():
        # 256 MB handed out without a begin_step(): ops driven directly in a loop (not through a model forward).  Every
        # earlier request was transient, so drain the device and start over.
        torch.cuda.synchronize()
        st["cursor"], st["zeroed"] = 0, 0
    if st["buf"] is None or st["cursor"] + npad > st["buf"].numel():
        if st["buf"] is not None:
            st["old"].append(st["buf"])
        size = max(npad * 2, 2 * (st["buf"].numel() if st["buf"] is not None else 0), 1 << 20)
        st["buf"] = torch.empty(size, device=device, dtype=torch.float32)
        st["cursor"], st["zeroed"] = 0, 0
        st["high"] = max(st["high"], 0)
    lo = st["cursor"]
    if lo + npad > st["zeroed"]:          # first step (or a new high-water mark): clear just this piece
        start = max(lo, st["zeroed"])
        call("deer_fill_zero", st["buf"].data_ptr() + 4 * start, lo + npad - start, None, 0)
        if start <= st["zeroed"]:
            st["zeroed"] = lo + npad
    st["cursor"] = lo + npad
    st["high"] = max(st["high"], st["cursor"])
    return st["buf"][lo:lo + n].view(*shape)


def set_gemm_engine(engine: int):
    """0 auto (tcgen05 where the shape allows), 1 fp32 SIMT everywhere, 2 force tcgen05 (raises if unsupported).
    The LSTM recurrence follows: SIMT -> exact fp32 stepwise; otherwise the TF32 engines."""
    _state["engine"] = int(engine)
    _state["lstm_engine"] = ENGINE_SIMT if int(engine) == ENGINE_SIMT else ENGINE_AUTO


def set_lstm_engine(engine: int):
    _state["lstm_engine"] = int(engine)


def set_exact_small_forward(on: bool, small_rows: int = 8192, backward: Optional[bool] = None,
                            small_rows_bwd: Optional[int] = None):
    """Precision policy of the time-batched contractions: below `small_rows` (forward) / `small_rows_bwd` (backward) rows
    they run on the fp32-grade engine, from there on the TF32 tcgen05 engine."""
    _state["exact_small_fwd"] = bool(on)
    _state["exact_small_bwd"] = bool(on if backward is None else backward)
    _state["small_rows"] = int(small_rows)
    _state["small_rows_bwd"] = int(small_rows if small_rows_bwd is None else small_rows_bwd)


def set_conv_exact(fwd: bool = False, bwd: bool = False):
    """Diagnostics: Conv1d taps (forward / backward GEMMs) on the fp32-grade engine through the im2col path."""
    _state["conv_exact"] = (1 if fwd else 0) | (2 if bwd else 0)


def _bwd_engine(M: int, chain: bool = False):
    """Engine for a backward GEMM of an nn.Linear with M rows; `chain`: see _fwd_engine."""
    if _state["engine"] == ENGINE_AUTO and _state["exact_small_bwd"] and (chain or M < _state["small_rows_bwd"]):
        return _state["exact_engine"]
    return None


def _fwd_engine(M: int, chain: bool = False):
    """Engine for a FORWARD nn.Linear with M rows under the precision policy.  `chain` = a post-pooling layer (one row
    per sample: fusion, NIG head, pooled model): exact at EVERY batch size -- the policy is keyed on the layer's role, not
    on the row count, so outputs do not change discontinuously with the batch.  Time-batched contractions (M = B*T
    rows: scorers, Conv1d taps, projections) use the TF32 tensor-core engine once M reaches `small_rows`."""
    if _state["engine"] == ENGINE_AUTO and _state["exact_small_fwd"] and (chain or M < _state["small_rows"]):
        return _state["exact_engine"]
    return None


def set_exact_engine(engine: int):
    """Engine of the fp32-grade contractions: ENGINE_X3 (default: error-compensated 3xTF32 tensor-core tiles with fused
    bias / activation / dropout / backward-gate / bias-gradient) or ENGINE_SIMT (fp32 FFMA tiles, separate elementwise
    kernels: the round-1 path, kept as the on-device reference)."""
    _state["exact_engine"] = int(engine)


def _fused_chain() -> bool:
    """The fused 3xTF32 Linear nodes are in use (default policy, no forced engine)."""
    return (_state["engine"] == ENGINE_AUTO and _state["exact_small_fwd"] and _state["exact_small_bwd"] and
            _state["exact_engine"] == ENGINE_X3)


def _req(t: torch.Tensor, name: str):
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise _lib.DeerError(f"deer_b200: `{name}` must be a CUDA tensor (no CPU fallback on this path)")
    if t.dtype != torch.float32:
        raise _lib.DeerError(f"deer_b200: `{name}` must be float32, got {t.dtype}")
    return t


def _rows2d(t: torch.Tensor):
    """View t [..., K] as a 2-D row matrix without copying when rows are evenly strided; returns (tensor, M, K, ld)."""
    K = t.shape[-1]
    if t.dim() == 2 and t.stride(1) == 1 and t.stride(0) >= K:
        return t, t.shape[0], K, t.stride(0)
    t2 = t.reshape(-1, K)
    if t2.stride(1) != 1 or (t2.shape[0] > 1 and t2.stride(0) < K):
        t2 = t2.contiguous()
    return t2, t2.shape[0], K, (t2.stride(0) if t2.shape[0] > 1 else K)


def gemm(A, lda, transA, B, ldb, transB, C, ldc, M, N, K, bias=None, act=0, beta=0.0, batch=1, sA=0, sB=0, sC=0,
         sBias=0, engine=None):
    call("deer_gemm", ptr(A) if isinstance(A, torch.Tensor) else A, lda, int(transA),
         ptr(B) if isinstance(B, torch.Tensor) else B, ldb, int(transB),
         ptr(C) if isinstance(C, torch.Tensor) else C, ldc, M, N, K, ptr(bias), act, float(beta), batch, sA, sB, sC,
         sBias, _state["engine"] if engine is None else engine)


def cast16(x: torch.Tensor, bf16: bool = False, pad_to: int = 8) -> torch.Tensor:
    """fp32 [..., K] -> fp16/bf16 [rows, Kp] shadow (Kp = K rounded up to `pad_to`, zero-filled) for deer_gemm_h16."""
    x2, M, K, ld = _rows2d(_req(x, "x"))
    Kp = (K + pad_to - 1) // pad_to * pad_to
    out = torch.empty((M, Kp), device=x.device, dtype=torch.bfloat16 if bf16 else torch.float16)
    call("deer_cast16", ptr(x2), ld, out.data_ptr(), Kp, M, K, Kp, int(bf16))
    return out


def _p16(t):
    return t.data_ptr() if isinstance(t, torch.Tensor) else t


def gemm_h16(A, lda, transA, B, ldb, transB, C, ldc, M, N, K, *, a_bf16=False, b_bf16=False, bias=None, act=0,
             beta=0.0, C16=None, ldc16=0, c16_bf16=False):
    """deer_gemm_h16: 16-bit operands (pointers or tensors), fp32 accumulate; fp32 output C, or (C=None) 16-bit C16."""
    call("deer_gemm_h16", _p16(A), lda, int(transA), int(a_bf16), _p16(B), ldb, int(transB), int(b_bf16),
         None if C is None else _p16(C), ldc, None if C16 is None else _p16(C16), ldc16, int(c16_bf16), M, N, K,
         ptr(bias), act, float(beta))


def cast_split16(x: torch.Tensor, rows=None, cols=None, ld=None, row_scale=None):
    """fp32 rows -> (hi, lo) FP16 [rows, Kp] with x = hi + lo to 22 significant bits (Kp = cols rounded up to 8).
    `x` may be a tensor (viewed as rows of its last dimension) or a raw (pointer, rows, cols, ld) description.
    `row_scale` [rows] (optional): every row is multiplied by its factor first (the text encoder's attention mask)."""
    if isinstance(x, torch.Tensor):
        x2, rows, cols, ld = _rows2d(_req(x, "x"))
        src, dev = ptr(x2), x.device
    else:
        src, dev = int(x[0]), x[1]
    Kp = (cols + 7) // 8 * 8
    hi = torch.empty((rows, Kp), device=dev, dtype=torch.float16)
    lo = torch.empty((rows, Kp), device=dev, dtype=torch.float16)
    call("deer_cast_split16", src, ld, ptr(row_scale), hi.data_ptr(), lo.data_ptr(), Kp, rows, cols, Kp)
    return hi, lo, Kp


def gemm_split(a_hi, a_lo, lda, b_hi, b_lo, ldb, C, ldc, M, N, K, bias=None, act=0):
    """C = act(A B^T + bias) on FP16 hi/lo operand pairs (deer_gemm_h16_split): A [M,K] rows (pitch lda, may be < K:
    overlapping windows), B [N,K] rows."""
    call("deer_gemm_h16_split", a_hi.data_ptr(), a_lo.data_ptr(), int(lda), 0, b_hi.data_ptr(), b_lo.data_ptr(),
         int(ldb), 1, ptr(C), int(ldc), int(M), int(N), int(K), ptr(bias), int(act))


def set_split_forward(on: bool, rows: int = 1024):
    """Time-batched FORWARD contractions with at least `rows` rows on the split-precision 16-bit engine (default on);
    off: TF32 tcgen05 from `small_rows` rows on (the round-1 policy; ~3e-4 forward error)."""
    _state["split_fwd"] = bool(on)
    _state["split_rows"] = int(rows)


def _split_fwd_ok(M: int, N: int, K: int, bias=None) -> bool:
    return (_state["split_fwd"] and _state["engine"] == ENGINE_AUTO and M >= _state["split_rows"] and M > 128 and
            N % 4 == 0 and N >= 64 and K >= 32)


def gemm_x3(A, lda, transA, B, ldb, transB, C, ldc, M, N, K, *, bias=None, act=0, beta=0.0, batch=1, sA=0, sB=0, sC=0,
            sBias=0, gate=None, ldgate=0, gate_mode=0, gate_scale=1.0, sGate=0, colsum=None, sColsum=0, drop=None,
            drop_ld=0, drop_col0=0, drop_batch_stride=0):
    """deer_gemm_x3: fused 3xTF32 GEMM (include/deer_b200.h).  Pointers or fp32 CUDA tensors; `drop` = (p, seed, offset,
    step tensor or None)."""
    def P(t):
        return None if t is None else (ptr(t) if isinstance(t, torch.Tensor) else int(t))
    a = _lib.GemmX3Args()
    a.A, a.B, a.C, a.bias, a.gate, a.colsum = P(A), P(B), P(C), P(bias), P(gate), P(colsum)
    a.lda, a.ldb, a.ldc, a.ldgate = int(lda), int(ldb), int(ldc), int(ldgate)
    a.sA, a.sB, a.sC, a.sBias, a.sGate, a.sColsum = int(sA), int(sB), int(sC), int(sBias), int(sGate), int(sColsum)
    if drop is not None and drop[0] > 0.0:
        a.drop_p, a.drop_seed, a.drop_offset = float(drop[0]), int(drop[1]), int(drop[2])
        a.drop_step = P(drop[3])
    a.drop_ld, a.drop_col0, a.drop_batch_stride = int(drop_ld), int(drop_col0), int(drop_batch_stride)
    a.M, a.N, a.K, a.batch = int(M), int(N), int(K), int(batch)
    a.transA, a.transB, a.act = int(transA), int(transB), int(act)
    a.beta = float(beta)
    a.gate_mode, a.gate_scale = int(gate_mode), float(gate_scale)
    _lib.check(_lib.load().deer_gemm_x3(a, _lib.stream()), "deer_gemm_x3")


_GATE_MODE = {1: 1, 2: 2, 3: 3}   # activation code -> gate mode (derivative from the saved output)


def _take_dropout(numel: int, p: float, training: bool):
    """Reserve the Philox block range of one dropout application: (p, seed, offset, step tensor) or None."""
    if not training or p <= 0.0:
        return None
    off = _dropout_state["offset"]
    _dropout_state["offset"] = off + (numel + 3) // 4
    return (float(p), _dropout_seed(), off, _dropout_state["step"])


def _colw(w: torch.Tensor, k0: int, k1: int):
    """Pointer/ld of the column block w[:, k0:k1] of a row-major weight."""
    return w.data_ptr() + 4 * k0, w.stride(0)


# ----------------------------------------------------------------------------------------------- Linear
class _Linear(torch.autograd.Function):
    """y = act(sum_i x_i W[:, blk_i]^T + b): nn.Linear applied to the (virtual) concatenation of the inputs."""

    @staticmethod
    def forward(ctx, w, b, act, n_in, *xs):
        _req(w, "weight")
        N, Ktot = w.shape
        rows = []
        k0 = 0
        y = None
        lead = xs[0].shape[:-1]
        chain = len(lead) == 1          # one row per sample: a post-pooling (fusion / head) layer, exact at every M
        for i, x in enumerate(xs):
            x2, M, K, ld = _rows2d(_req(x, "input"))
            if y is None:
                y = torch.empty((M, N), device=w.device, dtype=torch.float32)
            last = i == len(xs) - 1
            if not chain and len(xs) == 1 and _split_fwd_ok(M, N, K):
                # time-batched forward projection: fp32-grade products on FP16 hi/lo operand pairs (see gemm_split)
                xh, xl, Kp = cast_split16(x2)
                wh, wl, _ = cast_split16(w)
                gemm_split(xh, xl, Kp, wh, wl, Kp, y, N, M, N, K, bias=b, act=act)
            else:
                gemm(x2, ld, 0, w.data_ptr() + 4 * k0, w.stride(0), 1, y, N, M, N, K,
                     bias=b if last else None, act=act if last else 0, beta=0.0 if i == 0 else 1.0,
                     engine=_fwd_engine(M, chain))
            rows.append((x2, ld, k0, K))
            k0 += K
        assert k0 == Ktot, f"input widths {k0} != weight in-features {Ktot}"
        ctx.act = act
        ctx.chain = chain
        ctx.has_bias = b is not None
        ctx.params = (w, b)
        ctx.meta = [(ld, k, K) for (_, ld, k, K) in rows]
        ctx.in_shapes = [x.shape for x in xs]
        ctx.save_for_backward(w, y if act != 0 else None, *[r[0] for r in rows])
        return y.view(*lead, N)

    @staticmethod
    def backward(ctx, dy):
        w, y, *xs = ctx.saved_tensors
        N, Ktot = w.shape
        dy2, M, _, ld_dy = _rows2d(dy if dy.is_contiguous() else dy.contiguous())
        pw, pb = ctx.params
        db, db_direct = _acc(pb) if (ctx.has_bias and ctx.needs_input_grad[1]) else (None, False)
        if ctx.act != 0:
            dz = torch.empty_like(dy2)
            call("deer_bias_act_bwd", ptr(dy2), ld_dy, ptr(y), N, ptr(dz), N, ptr(db), M, N, ctx.act)
        else:
            dz = dy2
            if db is not None:
                call("deer_bias_act_bwd", ptr(dy2), ld_dy, None, 0, None, 0, ptr(db), M, N, 0)
        dw, dw_direct = _acc(pw) if ctx.needs_input_grad[0] else (None, False)
        # Trainer mode, small layers (the serial fusion / head chain, M = batch rows): dW is not needed before the
        # optimizer, so it leaves the dz -> dx critical path and runs on the weight-gradient stream, beside the
        # next layers' dx GEMMs (each of these kernels fills a fraction of the machine); the trainer joins the
        # stream before the gradient exchange (join_wgrad_stream).
        defer = (dw is not None and dw_direct and _state["defer_wgrad"] and M < _state["small_rows"] and dz.is_cuda)
        chain = ctx.chain
        if not chain and len(xs) == 1 and _bwd16_ok(M) and N % 8 == 0:
            # time-batched layer: BF16 operands on the 16-bit tcgen05 engine (dz cast once, shared by dW and dx)
            ld, k0, K = ctx.meta[0]
            dzb = cast16(dz, bf16=True)
            dxs = [None]
            if ctx.needs_input_grad[4]:
                wb = cast16(w, bf16=True)
                dx = torch.empty((M, K), device=w.device, dtype=torch.float32)
                gemm_h16(dzb, N, 0, wb, wb.shape[1], 0, dx, K, M, K, N, a_bf16=True, b_bf16=True)
                dxs = [dx.view(ctx.in_shapes[0])]
            if dw is not None:
                xb = cast16(xs[0], bf16=True)
                gemm_h16(dzb, N, 1, xb, xb.shape[1], 0, dw, Ktot, N, K, M, a_bf16=True, b_bf16=True, beta=1.0)
            return (None if dw_direct else dw, None if db_direct else db, None, None, *dxs)
        dxs = []
        for i, x2 in enumerate(xs):
            ld, k0, K = ctx.meta[i]
            if ctx.needs_input_grad[4 + i]:
                dx = torch.empty((M, K), device=w.device, dtype=torch.float32)
                gemm(dz, N, 0, w.data_ptr() + 4 * k0, w.stride(0), 0, dx, K, M, K, N, engine=_bwd_engine(M, chain))
                dxs.append(dx.view(ctx.in_shapes[i]))
            else:
                dxs.append(None)
            if dw is not None and not defer:
                gemm(dz, N, 1, x2, ld, 0, dw.data_ptr() + 4 * k0, Ktot, N, K, M, beta=1.0,
                     engine=_bwd_engine(M, chain))
        if defer:
            cur = torch.cuda.current_stream()
            aux = _wgrad_stream()
            aux.wait_stream(cur)
            with torch.cuda.stream(aux):
                for i, x2 in enumerate(xs):
                    ld, k0, K = ctx.meta[i]
                    gemm(dz, N, 1, x2, ld, 0, dw.data_ptr() + 4 * k0, Ktot, N, K, M, beta=1.0,
                         engine=_bwd_engine(M, chain))
                    x2.record_stream(aux)
            dz.record_stream(aux)
            _wgrad["pending"] = True
        return (None if dw_direct else dw, None if db_direct else db, None, None, *dxs)


class _LinearX3(torch.autograd.Function):
    """y = dropout(act(sum_i x_i W[:, blk_i]^T + b)) as ONE launch per input block, backward as two launches per block:
    the fused 3xTF32 engine (csrc/gemm_x3.cu) applies bias / activation / inverted dropout in the epilogue, the
    ReLU-and-dropout (or tanh / sigmoid) derivative while it reads dy ("gate" from the saved output: d > 0 <=> the unit
    was active AND kept), and the bias gradient as the column sums of the gated dy inside the dW GEMM."""

    @staticmethod
    def forward(ctx, w, b, act, drop, n_in, *xs):
        _req(w, "weight")
        N, Ktot = w.shape
        rows = []
        k0 = 0
        y = None
        lead = xs[0].shape[:-1]
        for i, x in enumerate(xs):
            x2, M, K, ld = _rows2d(_req(x, "input"))
            if y is None:
                y = torch.empty((M, N), device=w.device, dtype=torch.float32)
            last = i == len(xs) - 1
            gemm_x3(x2, ld, 0, w.data_ptr() + 4 * k0, w.stride(0), 1, y, N, M, N, K, bias=b if last else None,
                    act=act if last else 0, beta=0.0 if i == 0 else 1.0, drop=drop if last else None)
            rows.append((x2, ld, k0, K))
            k0 += K
        assert k0 == Ktot, f"input widths {k0} != weight in-features {Ktot}"
        ctx.act = act
        ctx.drop_p = drop[0] if drop is not None else 0.0
        ctx.has_bias = b is not None
        ctx.params = (w, b)
        ctx.meta = [(ld, k, K) for (_, ld, k, K) in rows]
        ctx.in_shapes = [x.shape for x in xs]
        ctx.save_for_backward(w, y if (act != 0 or ctx.drop_p > 0.0) else None, *[r[0] for r in rows])
        return y.view(*lead, N)

    @staticmethod
    def backward(ctx, dy):
        w, y, *xs = ctx.saved_tensors
        N, Ktot = w.shape
        dy2, M, _, ld_dy = _rows2d(dy if dy.is_contiguous() else dy.contiguous())
        pw, pb = ctx.params
        gate, gmode, gscale = None, 0, 1.0
        if y is not None:
            gate, gmode = y, _GATE_MODE[ctx.act]
            gscale = 1.0 / (1.0 - ctx.drop_p) if ctx.drop_p > 0.0 else 1.0
        need_db = ctx.has_bias and ctx.needs_input_grad[1]
        need_dw = ctx.needs_input_grad[0]
        db, db_direct = _acc(pb) if need_db else (None, False)
        dw, dw_direct = _acc(pw) if need_dw else (None, False)
        if need_db and not need_dw:        # (not on the model's path: the bias gradient rides on the dW GEMM)
            dz = torch.empty_like(dy2)
            call("deer_bias_act_bwd", ptr(dy2), ld_dy, ptr(y), N, ptr(dz), N, ptr(db), M, N, ctx.act)
        defer = (dw is not None and dw_direct and (db is None or db_direct) and _state["defer_wgrad"] and
                 M < _state["small_rows"])
        dxs = []
        for i, x2 in enumerate(xs):
            ld, k0, K = ctx.meta[i]
            if ctx.needs_input_grad[5 + i]:
                dx = torch.empty((M, K), device=w.device, dtype=torch.float32)
                gemm_x3(dy2, ld_dy, 0, w.data_ptr() + 4 * k0, w.stride(0), 0, dx, K, M, K, N, gate=gate, ldgate=N,
                        gate_mode=gmode, gate_scale=gscale)
                dxs.append(dx.view(ctx.in_shapes[i]))
            else:
                dxs.append(None)

        def wgrads():
            for i, x2 in enumerate(xs):
                ld, k0, K = ctx.meta[i]
                gemm_x3(dy2, ld_dy, 1, x2, ld, 0, dw.data_ptr() + 4 * k0, Ktot, N, K, M, beta=1.0, gate=gate, ldgate=N,
                        gate_mode=gmode, gate_scale=gscale, colsum=db if (i == 0 and need_db) else None)

        if dw is not None:
            if defer:
                # trainer mode: dW (+ db) is not needed before the optimizer, so it leaves the dy -> dx critical path and
                # runs on the weight-gradient stream beside the next layers' dx GEMMs (joined before the exchange)
                cur = torch.cuda.current_stream()
                aux = _wgrad_stream()
                aux.wait_stream(cur)
                with torch.cuda.stream(aux):
                    wgrads()
                    for x2 in xs:
                        x2.record_stream(aux)
                dy2.record_stream(aux)
                if gate is not None:
                    gate.record_stream(aux)
                _wgrad["pending"] = True
            else:
                wgrads()
        return (None if dw_direct else dw, None if db_direct else db, None, None, None, *dxs)


def linear(x, w, b=None, act="none", dropout: float = 0.0, training: bool = False):
    """nn.Linear (+ activation) (+ nn.Dropout) on x, or on the virtual concatenation of a list of inputs.  Post-pooling
    layers (2-D inputs: one row per sample) run as one fused 3xTF32 launch (`_LinearX3`) under the default policy;
    time-batched layers and forced engines take the generic node with separate elementwise kernels."""
    xs = x if isinstance(x, (list, tuple)) else [x]
    a = ACT[act]
    if xs[0].dim() == 2 and _fused_chain() and (dropout <= 0.0 or not training or a == 1):
        drop = _take_dropout(xs[0].shape[0] * w.shape[0], dropout, training)
        return _LinearX3.apply(w, b, a, drop, len(xs), *xs)
    y = _Linear.apply(w, b, a, len(xs), *xs)
    return _apply_dropout(y, dropout, training)


# ----------------------------------------------------------------------------------------------- LayerNorm
class _LayerNorm(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, g, b, eps):
        x2, M, N, ld = _rows2d(_req(x, "input"))
        if ld != N:
            x2 = x2.contiguous()
        y = torch.empty((M, N), device=x.device, dtype=torch.float32)
        mean = torch.empty(M, device=x.device, dtype=torch.float32)
        rstd = torch.empty(M, device=x.device, dtype=torch.float32)
        call("deer_layernorm_fwd", ptr(x2), ptr(g), ptr(b), ptr(y), ptr(mean), ptr(rstd), M, N, float(eps))
        ctx.save_for_backward(x2, g, mean, rstd)
        ctx.shape = x.shape
        ctx.params = (g, b)
        return y.view(x.shape)

    @staticmethod
    def backward(ctx, dy):
        x2, g, mean, rstd = ctx.saved_tensors
        M, N = x2.shape
        dy2 = dy.reshape(M, N)
        if not dy2.is_contiguous():
            dy2 = dy2.contiguous()
        dx = torch.empty_like(x2)
        dg, dg_direct = _acc(ctx.params[0])
        db, db_direct = _acc(ctx.params[1])
        call("deer_layernorm_bwd", ptr(dy2), ptr(x2), ptr(g), ptr(mean), ptr(rstd), ptr(dx), ptr(dg), ptr(db), M, N)
        return dx.view(ctx.shape), None if dg_direct else dg, None if db_direct else db, None


def layer_norm(x, g, b, eps=1e-5):
    return _LayerNorm.apply(x, g, b, eps)


# ----------------------------------------------------------------------------------------------- Dropout
_dropout_state = {"seed": 0x5EED, "offset": 0, "step": None, "host_step": 0}
_SEED_MIX = 0x9E3779B97F4A7C15


def manual_seed(seed: int):
    _dropout_state["seed"] = int(seed)
    _dropout_state["offset"] = 0
    _dropout_state["host_step"] = 0


def set_dropout_step_tensor(t: Optional[torch.Tensor]):
    """int64 CUDA scalar a trainer increments once per step; mixed into the Philox counter so CUDA-graph replays
    draw fresh masks.  None disables it (the host-side step counter of begin_step() is used instead).  Returns the
    previous binding: a trainer binds its own tensor around its step and restores the caller's afterwards, so two
    trainers in one process never share masks."""
    prev = _dropout_state["step"]
    _dropout_state["step"] = t
    return prev


def begin_step():
    """Once per model forward: restart the per-step element offsets (graph capture and eager agree) and advance the
    host-side step counter that keys the masks when no device step tensor is bound -- a plain torch.optim loop around
    the drop-in modules draws fresh dropout masks every forward."""
    _dropout_state["offset"] = 0
    _dropout_state["host_step"] += 1
    _arena_begin_step()


def _dropout_seed() -> int:
    """Seed of the masks drawn now: the base seed, mixed with the host step unless a device step tensor is bound."""
    if _dropout_state["step"] is not None:
        return _dropout_state["seed"]
    return (_dropout_state["seed"] ^ (_dropout_state["host_step"] * _SEED_MIX)) & 0xFFFFFFFFFFFFFFFF


class _Dropout(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, p, seed, offset):
        xc = _req(x, "input").contiguous()
        y = torch.empty_like(xc)
        st = _dropout_state["step"]
        call("deer_dropout", ptr(xc), ptr(y), xc.numel(), float(p), seed, offset, ptr(st))
        ctx.p, ctx.seed, ctx.offset, ctx.step = p, seed, offset, st
        return y

    @staticmethod
    def backward(ctx, dy):
        dyc = dy.contiguous()
        dx = torch.empty_like(dyc)
        call("deer_dropout", ptr(dyc), ptr(dx), dyc.numel(), float(ctx.p), ctx.seed, ctx.offset, ptr(ctx.step))
        return dx, None, None, None


def dropout(x, p: float, training: bool):
    if not training or p <= 0.0:
        return x
    off = _dropout_state["offset"]
    _dropout_state["offset"] = off + (x.numel() + 3) // 4
    return _Dropout.apply(x, p, _dropout_seed(), off)


_apply_dropout = dropout


# ----------------------------------------------------------------------------------------------- attention pooling
class _RowDot(torch.autograd.Function):
    @staticmethod
    def forward(ctx, h, w, b):
        h2, M, N, ld = _rows2d(_req(h, "hidden"))
        if ld != N:
            h2 = h2.contiguous()
        s = torch.empty(M, device=h.device, dtype=torch.float32)
        call("deer_rowdot_fwd", ptr(h2), ptr(w), ptr(b), ptr(s), M, N)
        ctx.save_for_backward(h2, w)
        ctx.shape = h.shape
        ctx.params = (w, b)
        return s.view(h.shape[:-1])

    @staticmethod
    def backward(ctx, ds):
        h2, w = ctx.saved_tensors
        M, N = h2.shape
        dsc = ds.reshape(M).contiguous()
        dh = torch.empty_like(h2)
        dw, dw_direct = _acc(ctx.params[0])
        db, db_direct = _acc(ctx.params[1])
        call("deer_rowdot_bwd", ptr(dsc), ptr(h2), ptr(w), ptr(dh), ptr(dw), ptr(db), M, N)
        return dh.view(ctx.shape), None if dw_direct else dw, None if db_direct else db


def rowdot(h, w, b):
    """s[...] = h[..., :] . w + b   (w is the [1,N] weight of a Linear(N,1), b its [1] bias)."""
    return _RowDot.apply(h, w, b)


def sequence_lengths(lengths, B: int, T: int, device) -> Optional[torch.Tensor]:
    """Per-utterance lengths [B] (int32 or int64; sample b is x[b, :L_b], frames t >= L_b are padding whose content does
    not matter) as the CUDA tensor the length-aware kernels read, in its own dtype (no conversion launch).  A CPU tensor
    (or a sequence) is validated here -- 1 <= L_b <= T, as pack_padded_sequence requires -- and copied to `device`.  A
    CUDA tensor is NOT read on the host (that would synchronise and break CUDA-graph capture of a step): the kernels
    clamp its values to [1, T].  None -> None."""
    if lengths is None:
        return None
    if not torch.is_tensor(lengths):
        lengths = torch.as_tensor(lengths)
    if lengths.dtype not in (torch.int32, torch.int64):
        raise _lib.DeerError(f"deer_b200: lengths must be an int32 or int64 tensor, got {lengths.dtype}")
    if tuple(lengths.shape) != (B,):
        raise _lib.DeerError(f"deer_b200: lengths must have shape [{B}], got {tuple(lengths.shape)}")
    if not lengths.is_cuda:
        if B > 0 and (int(lengths.min()) < 1 or int(lengths.max()) > T):
            raise _lib.DeerError(f"deer_b200: lengths must lie in [1, {T}] (got {int(lengths.min())} .. "
                                 f"{int(lengths.max())})")
        lengths = lengths.to(device)
    return lengths.contiguous()


def _len_i64(lengths: torch.Tensor) -> int:
    return int(lengths.dtype == torch.int64)


def _pool_fwd(x, xs_b, xs_t, s, ss_b, ss_t, m, lengths, out, wts, B, T, D, premask=False):
    """Attention pooling forward over each sample's frames t < L_b (lengths) or over all T (mask m / premask)."""
    if lengths is not None:
        call("deer_attn_pool_len_fwd", ptr(x), xs_b, xs_t, ptr(s), ss_b, ss_t, lengths.data_ptr(), _len_i64(lengths),
             ptr(out), ptr(wts), B, T, D)
    else:
        call("deer_attn_pool_fwd", ptr(x), xs_b, xs_t, ptr(s), ss_b, ss_t, ptr(m), ptr(out), ptr(wts), B, T, D,
             int(premask))


def _pool_bwd(dout, x, xs_b, xs_t, s, ss_b, ss_t, m, lengths, wts, dx, ds, B, T, D, premask=False):
    """Attention pooling backward, dx overwritten (None: not produced); with lengths dx and ds are 0 at padded rows."""
    if lengths is not None:
        call("deer_attn_pool_len_bwd", ptr(dout), ptr(x), xs_b, xs_t, ss_b, ss_t, lengths.data_ptr(), _len_i64(lengths),
             ptr(wts), ptr(dx), ptr(ds), B, T, D)
    else:
        call("deer_attn_pool_bwd", ptr(dout), ptr(x), xs_b, xs_t, ptr(s), ss_b, ss_t, ptr(m), ptr(wts), ptr(dx), ptr(ds),
             B, T, D, 0, int(premask))


class _AttnPool(torch.autograd.Function):
    """x [B,T,D] (any b/t strides, unit d stride), scores s [B,T] (any strides), mask [B,T] or None."""

    @staticmethod
    def forward(ctx, x, s, mask, lengths=None):
        _req(x, "x"), _req(s, "scores")
        B, T, D = x.shape
        if x.stride(2) != 1:
            x = x.contiguous()
        m = None if mask is None else _req(mask, "mask").contiguous()
        if lengths is not None and m is not None:
            raise _lib.DeerError("deer_b200: attn_pool takes a mask or lengths, not both")
        out = torch.empty((B, D), device=x.device, dtype=torch.float32)
        wts = torch.empty((B, T), device=x.device, dtype=torch.float32)
        ctx.lengths = lengths
        _pool_fwd(x, x.stride(0), x.stride(1), s, s.stride(0), s.stride(1), m, lengths, out, wts, B, T, D)
        ctx.save_for_backward(x, s, m, wts)
        ctx.mark_non_differentiable(wts)
        return out, wts

    @staticmethod
    def backward(ctx, dout, _dw):
        x, s, m, wts = ctx.saved_tensors
        B, T, D = x.shape
        dx = torch.empty_strided(x.shape, x.stride(), device=x.device, dtype=torch.float32)
        ds = torch.empty_strided(s.shape, s.stride(), device=x.device, dtype=torch.float32)
        _pool_bwd(dout.contiguous(), x, x.stride(0), x.stride(1), s, s.stride(0), s.stride(1), m, ctx.lengths, wts, dx, ds,
                  B, T, D)
        ctx.lengths = None
        return dx, ds, None, None


def attn_pool(x, s, mask=None, lengths=None):
    """`lengths`: per-utterance lengths (sequence_lengths): softmax and sum over t < L_b only, 0 weight elsewhere."""
    return _AttnPool.apply(x, s, mask, lengths)


class _ScorerPool(torch.autograd.Function):
    """Attention pooling with its Linear-Tanh-Linear scorer as ONE autograd node (encoders.py:93-98,383-384; :462-467,
    543-544; :597-602,738-746):  s = w2 . tanh(x W1^T + b1) + b2;  p = softmax_t(s) [masked, renormalised];
    out[b] = sum_t p[b,t] x[b,t].  x [R0,R1,D] contiguous enumerates (t,b) (time_major) or (b,t).
    x feeds both the scorer and the weighted sum; as two nodes autograd materialised both input gradients and added
    them with a separate kernel (157 MB at the audio encoder).  Here the pooling backward writes dx and the scorer's
    input-gradient GEMM accumulates onto it (beta = 1)."""

    @staticmethod
    def forward(ctx, x, w1, b1, w2, b2, mask, time_major, precise=True, x_bf16=None, premask=False, lengths=None):
        """x_bf16: optional BF16 copy of x written by its producer (the LSTM recurrence kernel's shadow of h): the B
        operand of dW1 in backward without a cast pass.
        premask: scorer and pooling see x~[b,t] = mask[b,t] x[b,t] (encoders.py:733-735: `token_embeddings *
        attention_mask`) -- applied inside the operand cast and the pooling kernels, the masked copy (50 MB read + write at
        B = 256) is never materialised.  Batch-major x only; the scorer then runs on the split-precision engine.
        lengths: per-utterance lengths [B] (sequence_lengths): the softmax and the weighted sum cover t < L_b only; the
        scorer still runs on every row, but padded rows get weight 0, ds = 0 and dx = 0, so the scorer's backward GEMMs
        take nothing from them."""
        x = _req(x, "x").contiguous()
        premask = bool(premask)
        if lengths is not None and (mask is not None or premask):
            raise _lib.DeerError("deer_b200: scorer_pool takes a mask or lengths, not both")
        ctx.lengths = lengths
        if premask and (mask is None or time_major or ctx.needs_input_grad[0] or not (precise and _split_fwd_ok(
                x.shape[0] * x.shape[1], w1.shape[0], x.shape[2]))):
            raise _lib.DeerError("deer_b200: scorer_pool(premask=True) needs a mask, batch-major x without gradient and a "
                                 "shape the split-precision engine takes")
        ctx.x_bf16 = (x_bf16 if (x_bf16 is not None and x_bf16.dtype == torch.bfloat16 and x_bf16.is_contiguous() and
                                 x_bf16.numel() == x.numel()) else None)
        R0, R1, D = x.shape
        M = R0 * R1
        Hd = w1.shape[0]
        dev = x.device
        B, T = (R1, R0) if time_major else (R0, R1)
        xs_b, xs_t = (D, B * D) if time_major else (T * D, D)
        ss_b, ss_t = (1, B) if time_major else (T, 1)
        hidden = torch.empty((M, Hd), device=dev, dtype=torch.float32)
        m = None if mask is None else _req(mask, "mask").contiguous()
        if precise and _split_fwd_ok(M, Hd, D):
            xh, xl, Kp = cast_split16(x.view(M, D), row_scale=m if premask else None)
            wh, wl, _ = cast_split16(w1)
            gemm_split(xh, xl, Kp, wh, wl, Kp, hidden, Hd, M, Hd, D, bias=b1, act=ACT["tanh"])
        else:
            gemm(x, D, 0, w1, w1.stride(0), 1, hidden, Hd, M, Hd, D, bias=b1, act=ACT["tanh"], engine=_fwd_engine(M))
        sc = torch.empty(M, device=dev, dtype=torch.float32)
        w2v = w2.reshape(-1)
        call("deer_rowdot_fwd", ptr(hidden), ptr(w2v), ptr(b2), ptr(sc), M, Hd)
        out = torch.empty((B, D), device=dev, dtype=torch.float32)
        wts = torch.empty((B, T), device=dev, dtype=torch.float32)
        _pool_fwd(x, xs_b, xs_t, sc, ss_b, ss_t, m, lengths, out, wts, B, T, D, premask)
        ctx.save_for_backward(x, hidden, sc, m, wts, w1, w2v)
        ctx.premask = premask
        ctx.geom = (B, T, D, M, Hd, xs_b, xs_t, ss_b, ss_t)
        ctx.params = (w1, b1, w2, b2)
        ctx.mark_non_differentiable(wts)
        ctx.set_materialize_grads(False)
        return out, wts

    @staticmethod
    def backward(ctx, dout, _dw):
        x, hidden, sc, m, wts, w1, w2v = ctx.saved_tensors
        B, T, D, M, Hd, xs_b, xs_t, ss_b, ss_t = ctx.geom
        dev = x.device
        pw1, pb1, pw2, pb2 = ctx.params
        need_dx = ctx.needs_input_grad[0]
        if dout is None:
            dout = torch.zeros((B, D), device=dev, dtype=torch.float32)
        dx = torch.empty_like(x) if need_dx else None    # an input tensor (text embeddings): only ds is produced
        ds = torch.empty(M, device=dev, dtype=torch.float32)
        doutc = dout.contiguous()
        # the pooling's own input gradient w[b,t] dout[b,:] inside the epilogue of the scorer's input-gradient GEMM (TF32
        # CTA-pair engine): the pooling kernel then writes no dx and the GEMM does not read it back (2 x 157 MB at the
        # audio encoder, in front of the BPTT of the last LSTM layer)
        time_major = xs_t != D
        rowterm = bool(need_dx and _state.get("pool_rowterm", True) and _state["engine"] == ENGINE_AUTO and
                       _bwd_engine(M) is None and not (_bwd16_ok(M) and Hd % 8 == 0 and D % 8 == 0) and
                       _lib.tf32_pair_on() and M > 256 and D >= 128 and D % 4 == 0 and Hd >= 64 and Hd % 4 == 0)
        # with lengths dx is written as 0 at padded rows (they become the dh the BPTT kernel reads); the GEMMs below add
        # exact zeros there (ds = 0 -> dh = 0), and the rowterm epilogue's w[b,t] dout[b] is 0 there too
        _pool_bwd(doutc, x, xs_b, xs_t, sc, ss_b, ss_t, m, ctx.lengths, wts, None if rowterm else dx, ds, B, T, D,
                  ctx.premask)
        ctx.lengths = None
        dw2, dw2_direct = _acc(pw2, like=w2v)
        db2, db2_direct = _acc(pb2)
        db1, db1_direct = _acc(pb1)
        # the whole scorer head backward in one pass over the saved tanh output
        dh = torch.empty_like(hidden)
        call("deer_scorer_bwd", ptr(ds), ptr(hidden), ptr(w2v), ptr(dh), ptr(dw2), ptr(db1), ptr(db2),
             ptr(m.view(-1)) if ctx.premask else None, M, Hd)
        dw1, dw1_direct = _acc(pw1)
        if _bwd16_ok(M) and Hd % 8 == 0 and D % 8 == 0:
            # BF16 operands on the 16-bit tcgen05 engine: dx += dh W1 (onto the pooling gradient), dW1 += dh^T x
            dhb = cast16(dh, bf16=True)
            if need_dx:
                wb = cast16(w1, bf16=True)
                gemm_h16(dhb, Hd, 0, wb, D, 0, dx, D, M, D, Hd, a_bf16=True, b_bf16=True, beta=1.0)
            xb = ctx.x_bf16 if ctx.x_bf16 is not None else cast16(x.view(M, D), bf16=True)
            gemm_h16(dhb, Hd, 1, xb, D, 0, dw1, D, Hd, D, M, a_bf16=True, b_bf16=True, beta=1.0)
        else:
            if rowterm:
                call("deer_gemm_rowterm", ptr(dh), Hd, 0, ptr(w1), w1.stride(0), 0, ptr(dx), D, M, D, Hd, ptr(wts), ptr(doutc),
                     B, T, int(time_major))
            elif need_dx:
                gemm(dh, Hd, 0, w1, w1.stride(0), 0, dx, D, M, D, Hd, beta=1.0, engine=_bwd_engine(M))
            if dw1_direct and _state["defer_wgrad"] and _state["direct_grad"]:
                # trainer mode: dW1 is not needed before the optimizer -- it leaves the path to the LSTM's BPTT and runs
                # on the weight-gradient stream (a split-K TF32 GEMM of 100 KB CTAs: it shares SMs with the recurrence)
                cur = torch.cuda.current_stream()
                aux = _wgrad_stream()
                aux.wait_stream(cur)
                with torch.cuda.stream(aux):
                    gemm(dh, Hd, 1, x, D, 0, dw1, D, Hd, D, M, beta=1.0, engine=_bwd_engine(M))
                dh.record_stream(aux)
                x.record_stream(aux)
                _wgrad["pending"] = True
            else:
                gemm(dh, Hd, 1, x, D, 0, dw1, D, Hd, D, M, beta=1.0, engine=_bwd_engine(M))
        ctx.x_bf16 = None
        return (dx if need_dx else None, None if dw1_direct else dw1, None if db1_direct else db1,
                None if dw2_direct else dw2.view_as(pw2), None if db2_direct else db2, None, None, None, None, None, None)


def set_pool_rowterm(on: bool):
    """Attention pooling's input gradient inside the epilogue of the scorer's input-gradient GEMM (default) or written by
    the pooling kernel and accumulated onto by the GEMM (ablation / reference point of the equality test)."""
    _state["pool_rowterm"] = bool(on)


def set_scorer_pool_fused(on: bool):
    """Scorer + attention pooling as one autograd node (default) or as separate Linear / rowdot / pooling nodes."""
    _state["scorer_pool_fused"] = bool(on)


def scorer_pool_fused() -> bool:
    return _state["scorer_pool_fused"]


def scorer_pool(x, w1, b1, w2, b2, mask=None, time_major=False, precise=True, x_bf16=None, premask=False, lengths=None):
    """(pooled [B,D], attention weights [B,T]) of x [T,B,D] (time_major) or [B,T,D]; see _ScorerPool.  `precise`: the
    scorer's forward GEMM on the split-precision engine (default); False = TF32 (the audio encoder: its pooled output
    averages 300 highly correlated steps and is dominated by the FP16 recurrence's own 4e-5, measured).
    `lengths`: per-utterance lengths (sequence_lengths): pooling over each sample's frames t < L_b only."""
    if premask:
        M = x.shape[0] * x.shape[1]
        if not (precise and _split_fwd_ok(M, w1.shape[0], x.shape[2])):
            # no split-precision engine for this shape (small batches, forced engines): materialise the masked rows
            x, premask = rowscale(x, mask), False
    return _ScorerPool.apply(x, w1, b1, w2, b2, mask, bool(time_major), bool(precise), x_bf16, bool(premask), lengths)


class _RowScale(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, mask):
        xc = _req(x, "x").contiguous()
        m = _req(mask, "mask").contiguous()
        D = xc.shape[-1]
        y = torch.empty_like(xc)
        call("deer_rowscale", ptr(xc), ptr(m), ptr(y), xc.numel() // D, D)
        ctx.save_for_backward(m)
        return y

    @staticmethod
    def backward(ctx, dy):
        (m,) = ctx.saved_tensors
        dyc = dy.contiguous()
        D = dyc.shape[-1]
        dx = torch.empty_like(dyc)
        call("deer_rowscale", ptr(dyc), ptr(m), ptr(dx), dyc.numel() // D, D)
        return dx, None


def rowscale(x, mask):
    return _RowScale.apply(x, mask)


def _mask_padding(x, lengths):
    B, T, D = x.shape
    y = torch.empty_like(x)
    call("deer_rowscale_len", ptr(x), ptr(y), lengths.data_ptr(), _len_i64(lengths), B, T, D)
    return y


class _MaskPadding(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, lengths):
        ctx.lengths = lengths
        return _mask_padding(x, lengths)

    @staticmethod
    def backward(ctx, dy):
        return _mask_padding(dy.contiguous(), ctx.lengths), None


def mask_padding(x, lengths):
    """x [B,T,D] with the padded frames t >= L_b (lengths: see sequence_lengths) replaced by zero rows, which are never
    read (NaN padding stays out).  An autograd node only when x needs a gradient; its backward is the same masked copy,
    so the input gradient is exactly 0 at padded frames."""
    x = _req(x, "x").contiguous()
    lengths = sequence_lengths(lengths, x.shape[0], x.shape[1], x.device)
    if x.requires_grad and torch.is_grad_enabled():
        return _MaskPadding.apply(x, lengths)
    return _mask_padding(x, lengths)


def linguistic_features(input_ids: torch.Tensor, attention_mask: torch.Tensor, max_length: int = 128) -> torch.Tensor:
    """EnhancedTextEncoder.extract_linguistic_features (encoders.py:648-699) as one integer kernel: [B,T] int64 token
    ids + mask -> [B,10] fp32 (no gradient path, as in the reference)."""
    if not (input_ids.is_cuda and attention_mask.is_cuda):
        raise _lib.DeerError("deer_b200: `input_ids` / `attention_mask` must be CUDA tensors (no CPU fallback)")
    if input_ids.dtype != torch.int64:
        raise _lib.DeerError(f"deer_b200: `input_ids` must be int64, got {input_ids.dtype}")
    if input_ids.shape != attention_mask.shape or input_ids.dim() != 2:
        raise _lib.DeerError("deer_b200: `input_ids` and `attention_mask` must both be [B,T]")
    ids = input_ids.contiguous()
    m = attention_mask.contiguous()
    if m.dtype != torch.int64:
        m = (m != 0).to(torch.int64)
    B, T = ids.shape
    out = torch.empty((B, 10), device=ids.device, dtype=torch.float32)
    if B > 0:
        call("deer_linguistic_features", ids.data_ptr(), m.data_ptr(), ptr(out), B, T, int(max_length))
    return out


class _PermuteBT(torch.autograd.Function):
    """[B,T,D] contiguous -> [T,B,D] contiguous."""

    @staticmethod
    def forward(ctx, x):
        xc = _req(x, "x").contiguous()
        B, T, D = xc.shape
        y = torch.empty((T, B, D), device=x.device, dtype=torch.float32)
        call("deer_permute_bt", ptr(xc), ptr(y), B, T, D)
        return y

    @staticmethod
    def backward(ctx, dy):
        dyc = dy.contiguous()
        T, B, D = dyc.shape
        dx = torch.empty((B, T, D), device=dy.device, dtype=torch.float32)
        call("deer_permute_bt", ptr(dyc), ptr(dx), T, B, D)
        return dx


def to_time_major(x):
    return _PermuteBT.apply(x)


def set_lstm_input_projection_fused(on: bool):
    """First LSTM layer's input projection inside the forward recurrence kernel (default) or as a 16-bit GEMM that writes
    FP16 pre-activations (ablation / reference point of the equality test)."""
    _state["lstm_xin"] = bool(on)


def set_lstm_defer_wgrad(on: bool):
    """Weight-gradient GEMMs of an LSTM layer that has another LSTM layer below it on the weight-gradient stream
    (trainer mode only; measured: no gain, 3.755 vs 3.747 ms) or in front of the lower layer's BPTT (default)."""
    _state["lstm_defer_wgrad"] = bool(on)


def set_lstm_dropout_mask(on: bool):
    """nn.LSTM's inter-layer dropout in backward: keep bits written by the forward pass and applied by the epilogue of
    the dx GEMM (default), or a Philox pass over dx (ablation / reference point of the equality test)."""
    _state["lstm_drop_mask"] = bool(on)


def set_lstm_batch_major_input(on: bool):
    """First LSTM layer reads the batch_first input through one permute + 16-bit cast pass (default) or through a
    materialised fp32 time-major copy (ablation / reference point of the equality test)."""
    _state["lstm_bm_input"] = bool(on)


# ----------------------------------------------------------------------------------------------- BiLSTM layer
class _BiLSTMLayer(torch.autograd.Function):
    """One bidirectional nn.LSTM layer on a time-major input x [T,B,I] -> h [T,B,2H]."""

    @staticmethod
    def forward(ctx, x, wif, whf, bif, bhf, wir, whr, bir, bhr, grad_mode=True):
        x = _req(x, "x").contiguous()
        T, B, In = x.shape
        H = whf.shape[1]
        dev = x.device
        keep = grad_mode and any(ctx.needs_input_grad)   # needs_input_grad ignores no_grad(): the caller's mode
        gates = torch.empty((T, B, 2, 4 * H), device=dev, dtype=torch.float32)
        bsum = torch.empty((2, 4 * H), device=dev, dtype=torch.float32)
        call("deer_axpby", ptr(bif), ptr(bhf), bsum.data_ptr(), 4 * H, 1.0, 1.0)
        call("deer_axpby", ptr(bir), ptr(bhr), bsum.data_ptr() + 16 * H, 4 * H, 1.0, 1.0)
        M = T * B
        for d, wi in enumerate((wif, wir)):
            gemm(x, In, 0, wi, wi.stride(0), 1, gates.data_ptr() + 16 * H * d, 8 * H, M, 4 * H, In,
                 bias=bsum[d])
        h = torch.empty((T, B, 2 * H), device=dev, dtype=torch.float32)
        whf_c, whr_c = whf.contiguous(), whr.contiguous()
        if keep:
            c_all = torch.empty((T, B, 2, H), device=dev, dtype=torch.float32)
            call("deer_lstm_fwd", ptr(gates), ptr(whf_c), ptr(whr_c), ptr(h), ptr(c_all), None, T, B, H,
                 _state["lstm_engine"])
            ctx.save_for_backward(x, wif, whf_c, wir, whr_c, gates, c_all, h)
        else:
            c_work = torch.empty((B, 2, H), device=dev, dtype=torch.float32)
            call("deer_lstm_fwd", ptr(gates), ptr(whf_c), ptr(whr_c), ptr(h), None, ptr(c_work), T, B, H,
                 _state["lstm_engine"])
        ctx.dims = (T, B, In, H)
        ctx.params = (wif, whf, bif, bhf, wir, whr, bir, bhr)
        return h

    @staticmethod
    def backward(ctx, dh):
        x, wif, whf, wir, whr, gates, c_all, h = ctx.saved_tensors
        T, B, In, H = ctx.dims
        dev = x.device
        dh = dh.contiguous()
        dh_work = torch.empty((B, 2, H), device=dev, dtype=torch.float32)
        dc_work = torch.empty((B, 2, H), device=dev, dtype=torch.float32)
        # gates is consumed: it becomes the pre-activation gradient buffer [T,B,2,4H]
        call("deer_lstm_bwd", ptr(gates), ptr(whf), ptr(whr), ptr(c_all), ptr(dh), ptr(dh_work), ptr(dc_work), T, B, H,
             _state["lstm_engine"])
        M = T * B
        G = 4 * H
        dx = None
        if ctx.needs_input_grad[0]:
            dx = torch.empty((T, B, In), device=dev, dtype=torch.float32)
            for d, wi in enumerate((wif, wir)):
                gemm(gates.data_ptr() + 4 * G * d, 2 * G, 0, wi, wi.stride(0), 0, dx, In, M, In, G,
                     beta=0.0 if d == 0 else 1.0)
        grads = []
        P = ctx.params
        for d, (wi, wh) in enumerate(((wif, whf), (wir, whr))):
            gp = gates.data_ptr() + 4 * G * d
            dwi, dwi_direct = _acc(P[4 * d], wi)
            gemm(gp, 2 * G, 1, x, In, 0, dwi, In, G, In, M, beta=1.0)
            dwh, dwh_direct = _acc(P[4 * d + 1], wh)
            if T > 1:
                Mr = (T - 1) * B
                if d == 0:   # rows t=1.. pair with h[t-1]
                    gemm(gp + 4 * B * 2 * G, 2 * G, 1, h.data_ptr(), 2 * H, 0, dwh, H, G, H, Mr, beta=1.0)
                else:        # rows t=..T-2 pair with h[t+1]
                    gemm(gp, 2 * G, 1, h.data_ptr() + 4 * (B * 2 * H + H), 2 * H, 0, dwh, H, G, H, Mr, beta=1.0)
            db = torch.zeros(G, device=dev, dtype=torch.float32)
            call("deer_bias_act_bwd", gp, 2 * G, None, 0, None, 0, ptr(db), M, G, 0)
            dbs = []
            for pb in (P[4 * d + 2], P[4 * d + 3]):   # b_ih and b_hh receive the same gradient
                tgt, direct = _acc(pb)
                if direct:
                    call("deer_axpby", ptr(db), ptr(tgt), ptr(tgt), G, 1.0, 1.0)
                    dbs.append(None)
                else:
                    dbs.append(db)
            grads.append((None if dwi_direct else dwi, None if dwh_direct else dwh, dbs[0], dbs[1]))
        (dwif, dwhf, dbif, dbhf), (dwir, dwhr, dbir, dbhr) = grads
        return dx, dwif, dwhf, dbif, dbhf, dwir, dwhr, dbir, dbhr, None


class _BiLSTMLayerCluster(torch.autograd.Function):
    """Same layer on the persistent 4-CTA-cluster kernels (csrc/lstm_cluster.cu, H == 256).

    The kernels read/write the gate dimension INTERLEAVED (column 4*unit+gate), so the input projection runs on
    row-interleaved copies of W_ih / (b_ih+b_hh) and the weight gradients computed from the interleaved dpre are
    un-interleaved (accumulating) into their targets.  The bias gradient comes out of the BPTT kernel itself.

    The five time-batched contractions of the layer (input projection, dx, dW_ih, dW_hh x2 directions) run on the
    16-bit tcgen05 engine (deer_gemm_h16): forward operands FP16 (same 11 significant bits as TF32 for these value
    ranges), backward operands BF16.  The LSTM kernels write the 16-bit shadows of h and dpre themselves; x and the
    weights are cast once per call.

    `drop` = (p, seed, offset) or None: nn.LSTM's inter-layer dropout on this layer's INPUT, fused into the 16-bit
    casts (the dropped fp32 tensor is never materialised) and into dx in backward."""

    @staticmethod
    def forward(ctx, x, wif, whf, bif, bhf, wir, whr, bir, bhr, drop=None, x16_in=None, emit_f16=False,
                grad_mode=True, batch_major=False, lengths=None):
        """x16_in: FP16 copy of x written by the previous layer's recurrence kernel (skips the cast pass); emit_f16: make
        this layer's kernel write such a copy of h.  Returns (h, h_f16 or an empty tensor).
        batch_major: x is the batch_first input [B,T,In] of the first layer (no gradient): one pass writes its
        time-major FP16 / BF16 operand copies (no fp32 time-major copy, no cast passes).
        lengths: per-utterance lengths [B] on the device (sequence_lengths) -- nn.LSTM on a packed sequence.  The input
        projection then runs as a GEMM (not inside the recurrence kernel), deer_lstm_mask_pre saturates the i / f / o
        gates of the padded rows of its output, and the recurrence and BPTT kernels run unchanged (DESIGN.md 4.12); the
        first layer's operand casts write zeros for padded frames."""
        x = _req(x, "x").contiguous()
        if batch_major:
            B, T, In = x.shape
        else:
            T, B, In = x.shape
        H = whf.shape[1]
        G = 4 * H
        dev = x.device
        keep = grad_mode and any(ctx.needs_input_grad)   # needs_input_grad ignores no_grad(): the caller's mode
        use16 = _state["lstm_gemm16"] and _state["engine"] == ENGINE_AUTO   # a forced engine (tests) is respected
        if lengths is not None and not use16:
            raise _lib.DeerError("deer_b200: LSTM lengths need the 16-bit GEMM path (engine AUTO)")
        b_il = torch.empty((2, G), device=dev, dtype=torch.float32)
        w16 = None
        if use16:
            # one pass: both directions' W_ih -> gate-interleaved FP16 [2G, Kp], b_ih + b_hh -> gate-interleaved [2G]
            Kp = (In + 7) // 8 * 8
            w16 = torch.empty((2 * G, Kp), device=dev, dtype=torch.float16)
            call("deer_lstm_prep", ptr(wif.contiguous()), ptr(wir.contiguous()), ptr(bif), ptr(bhf), ptr(bir), ptr(bhr),
                 w16.data_ptr(), ptr(b_il), H, In, Kp, 0)
            wi_il = torch.empty(0, device=dev, dtype=torch.float32)
        else:
            wi_il = torch.empty((2, G, In), device=dev, dtype=torch.float32)
            bsum = torch.empty(G, device=dev, dtype=torch.float32)
            for d, (wi, bi, bh) in enumerate(((wif, bif, bhf), (wir, bir, bhr))):
                call("deer_gate_rows_interleave", ptr(wi.contiguous()), ptr(wi_il[d]), H, In, 0, 0)
                call("deer_axpby", ptr(bi), ptr(bh), ptr(bsum), G, 1.0, 1.0)
                call("deer_gate_rows_interleave", ptr(bsum), ptr(b_il[d]), H, 1, 0, 0)
        M = T * B
        # FP16 pre-activations (16-bit GEMM epilogue -> LSTM kernel): the projection is bound by its output stream, and
        # the rounding (2^-12 relative, once) is of the order of what the FP16 operands already contribute
        pre16 = use16 and _state["lstm_pre16"] and M > 128
        # first layer (In <= 128): the input projection runs INSIDE the recurrence kernel (deer_lstm_cluster_fwd_xin) -- no
        # projection GEMM, no pre-activation tensor
        xin = bool(use16 and pre16 and drop is None and lengths is None and _state.get("lstm_xin", True) and
                   _lib.load().deer_lstm_cluster_xin_mode(B, int(keep), (In + 7) // 8 * 8) > 0)
        pre = None if xin else torch.empty((T, B, 2, G), device=dev, dtype=torch.float16 if pre16 else torch.float32)
        x16 = None
        if drop is not None and not (use16 and In % 8 == 0):
            raise _lib.DeerError("deer_b200: fused input dropout needs the 16-bit GEMM path and In % 8 == 0")
        ctx.drop = drop
        ctx.drop_step = _dropout_state["step"]
        ctx.xdrop_b16 = None
        ctx.drop_mask = None
        # the 16-bit shadow outputs are non-differentiable: without this autograd hands backward a zero-filled tensor
        # for each of them (a 79 MB BF16 fill per layer and step)
        ctx.set_materialize_grads(False)
        if batch_major and not (use16 and drop is None and not ctx.needs_input_grad[0]):
            raise _lib.DeerError("deer_b200: batch_major LSTM input needs the 16-bit GEMM path, no input dropout and an "
                                 "input without gradient")
        if use16:
            shadow16 = (x16_in is not None and x16_in.dtype == torch.float16 and x16_in.numel() == M * In and In % 8 == 0
                        and x16_in.is_contiguous())
            if batch_major or (lengths is not None and drop is None and not shadow16):
                # (permute +) both 16-bit casts in one pass over x: the FP16 operand and (training) the BF16 one of dW_ih;
                # with lengths, zeros for padded frames: a NaN / Inf in the padding of an input never reaches the
                # projection or dW_ih = dpre^T x
                x16 = torch.empty((M, Kp), device=dev, dtype=torch.float16)
                xb16 = torch.empty((M, Kp), device=dev, dtype=torch.bfloat16) if keep else None
                if lengths is not None:
                    call("deer_permute_bt_cast16_len", ptr(x), x16.data_ptr(), None if xb16 is None else xb16.data_ptr(),
                         lengths.data_ptr(), _len_i64(lengths), B, T, In, Kp, int(not batch_major))
                else:
                    call("deer_permute_bt_cast16", ptr(x), x16.data_ptr(), None if xb16 is None else xb16.data_ptr(),
                         B, T, In, Kp)
                ctx.xdrop_b16 = xb16
            elif drop is not None:                            # dropout + fp16 cast in one pass over x
                x16 = torch.empty((M, In), device=dev, dtype=torch.float16)
                # training: the same pass also writes the BF16 copy the weight-gradient GEMM of backward reads (79 MB
                # more to store here, instead of a second Philox pass over x in backward: 47 us -> ~10 us)
                xdrop_b16 = torch.empty((M, In), device=dev, dtype=torch.bfloat16) if keep else None
                # ... and the keep bits (1 bit per element): the epilogue of backward's dx GEMM applies them, instead of a
                # Philox read-modify-write pass over dx (56 us at B = 256)
                kmask = None
                if (keep and ctx.needs_input_grad[0] and _state.get("lstm_drop_mask", True) and M > 128 and In % 32 == 0
                        and (M * In) % 128 == 0):
                    kmask = torch.empty(M * In // 32, device=dev, dtype=torch.int32)
                call("deer_dropout_cast16", ptr(x), x16.data_ptr(), None if xdrop_b16 is None else xdrop_b16.data_ptr(),
                     M * In, float(drop[0]), drop[1], drop[2], ptr(ctx.drop_step),
                     None if kmask is None else kmask.data_ptr())
                ctx.xdrop_b16 = xdrop_b16
                ctx.drop_mask = kmask
            elif shadow16:
                x16 = x16_in.view(M, In)                      # the producer kernel's FP16 shadow: no cast pass
            else:
                x16 = cast16(x)                               # [M, Kp] fp16
            assert x16.shape[1] == Kp
            # both directions in ONE contraction: pre[M, 2G] = x16 [M, Kp] . w16[2G, Kp]^T (full 8 KB output rows)
            if xin:
                pass
            elif pre16:
                gemm_h16(x16, Kp, 0, w16, Kp, 1, None, 0, M, 2 * G, In, bias=b_il.view(-1), C16=pre, ldc16=2 * G)
            else:
                gemm_h16(x16, Kp, 0, w16, Kp, 1, pre, 2 * G, M, 2 * G, In, bias=b_il.view(-1))
            if lengths is not None:
                call("deer_lstm_mask_pre", pre.data_ptr(), int(pre16), lengths.data_ptr(), _len_i64(lengths), T, B, H)
        else:
            for d in range(2):
                gemm(x, In, 0, wi_il[d], In, 1, pre.data_ptr() + 4 * G * d, 2 * G, M, G, In, bias=b_il[d])
        h = torch.empty((T, B, 2 * H), device=dev, dtype=torch.float32)
        h16 = torch.empty((T, B, 2 * H), device=dev, dtype=torch.float16) if emit_f16 else None
        h16p = None if h16 is None else h16.data_ptr()
        whf_c, whr_c = whf.contiguous(), whr.contiguous()
        fwd_fn = "deer_lstm_cluster_fwd_pre16" if pre16 else "deer_lstm_cluster_fwd"
        if keep:
            Bp = (B + 31) // 32 * 32
            kdt = torch.float16 if _state["lstm_keep16"] else torch.float32     # DEER_OPT_LSTM_KEEP16
            gact = torch.empty(T * 2 * Bp * G, device=dev, dtype=kdt)
            c_blk = torch.empty(T * 2 * Bp * H, device=dev, dtype=kdt)
            hb16 = torch.empty((T, B, 2 * H), device=dev, dtype=torch.bfloat16) if use16 else None
            if xin:
                call("deer_lstm_cluster_fwd_xin", x16.data_ptr(), Kp, w16.data_ptr(), ptr(b_il), ptr(whf_c), ptr(whr_c), ptr(h),
                     ptr(gact), ptr(c_blk), h16p, None if hb16 is None else hb16.data_ptr(), T, B, H)
            else:
                call(fwd_fn, pre.data_ptr(), ptr(whf_c), ptr(whr_c), ptr(h), ptr(gact), ptr(c_blk), h16p,
                     None if hb16 is None else hb16.data_ptr(), T, B, H)
            ctx.save_for_backward(x, wi_il, whf_c, whr_c, gact, c_blk, h)
            # the fp32 pre buffer doubles as the fp32 dpre buffer; on the 16-bit path BPTT only writes the BF16 dpre
            ctx.pre = None if use16 else pre
            ctx.hb16 = hb16
        elif xin:
            call("deer_lstm_cluster_fwd_xin", x16.data_ptr(), Kp, w16.data_ptr(), ptr(b_il), ptr(whf_c), ptr(whr_c), ptr(h),
                 None, None, h16p, None, T, B, H)
        else:
            call(fwd_fn, pre.data_ptr(), ptr(whf_c), ptr(whr_c), ptr(h), None, None, h16p, None, T, B, H)
        ctx.dims = (T, B, In, H)
        ctx.use16 = use16
        ctx.params = (wif, whf, bif, bhf, wir, whr, bir, bhr)
        if h16 is None:
            h16 = torch.empty(0, device=dev, dtype=torch.float16)
        hb_out = ctx.hb16 if (keep and ctx.hb16 is not None) else torch.empty(0, device=dev, dtype=torch.bfloat16)
        ctx.mark_non_differentiable(h16, hb_out)
        return h, h16, hb_out

    @staticmethod
    def backward(ctx, dh, _dh16=None, _dhb16=None):
        x, wi_il, whf, whr, gact, c_blk, h = ctx.saved_tensors
        T, B, In, H = ctx.dims
        G = 4 * H
        dev = x.device
        dh = torch.zeros((T, B, 2 * H), device=dev, dtype=torch.float32) if dh is None else dh.contiguous()
        dpre = ctx.pre
        hb16 = ctx.hb16
        ctx.pre = ctx.hb16 = None
        use16 = ctx.use16
        M = T * B
        if use16:   # the three gate-interleaved gradient accumulators of the layer in one zero-filled allocation
            zbuf = zeros_scratch(2 * G * (In + H + 1), dev)
            dwi_il2 = zbuf[:2 * G * In].view(2, G, In)
            dwh_il2 = zbuf[2 * G * In:2 * G * (In + H)].view(2, G, H)
            db_il = zbuf[2 * G * (In + H):].view(2, G)
        else:
            db_il = zeros_scratch((2, G), dev)
        dpre16 = torch.empty((T, B, 2, G), device=dev, dtype=torch.bfloat16) if use16 else None
        call("deer_lstm_cluster_bwd", ptr(gact), ptr(c_blk), ptr(dh), ptr(whf), ptr(whr),
             None if dpre is None else ptr(dpre), ptr(db_il), None if dpre16 is None else dpre16.data_ptr(), T, B, H)
        dx = None
        drop = ctx.drop
        if use16:
            if ctx.xdrop_b16 is not None:
                xb16 = ctx.xdrop_b16                           # written by the forward's (dropout / permute) + cast pass
                ctx.xdrop_b16 = None
            elif drop is not None:                             # the same mask, regenerated while casting to bf16
                xb16 = torch.empty((M, In), device=dev, dtype=torch.bfloat16)
                call("deer_dropout_cast16", ptr(x), None, xb16.data_ptr(), M * In, float(drop[0]), drop[1], drop[2],
                     ptr(ctx.drop_step))
            else:
                xb16 = cast16(x, bf16=True)                    # [M, Kp] bf16: B operand of dW_ih (MN-major)
            Kp = xb16.shape[1]
            if ctx.needs_input_grad[0]:
                # [2G, Kp] bf16 gate-interleaved W_ih of both directions: B operand of dx (MN-major [K=G, N=In])
                wb16 = torch.empty((2 * G, Kp), device=dev, dtype=torch.bfloat16)
                call("deer_lstm_prep", ptr(ctx.params[0].contiguous()), ptr(ctx.params[4].contiguous()), None, None, None,
                     None, wb16.data_ptr(), None, H, In, Kp, 1)
                dx = torch.empty((T, B, In), device=dev, dtype=torch.float32)
                # dx = dpre16 [M, 2G] . wb16 [2G, In]: the sum over the two directions is the K = 2G contraction itself
                kmask = ctx.drop_mask
                ctx.drop_mask = None
                if drop is not None and kmask is not None:
                    # d/dx of the input dropout inside the GEMM's epilogue (keep bits written by the forward pass)
                    call("deer_gemm_h16_dropmask", dpre16.data_ptr(), 2 * G, 0, 1, wb16.data_ptr(), Kp, 0, 1, ptr(dx), In,
                         M, In, 2 * G, kmask.data_ptr(), 1.0 / (1.0 - float(drop[0])))
                else:
                    gemm_h16(dpre16, 2 * G, 0, wb16, Kp, 0, dx, In, M, In, 2 * G, a_bf16=True, b_bf16=True, beta=0.0)
                    if drop is not None:                       # d/dx of the input dropout, in place
                        call("deer_dropout", ptr(dx), ptr(dx), dx.numel(), float(drop[0]), drop[1], drop[2],
                             ptr(ctx.drop_step))
        elif ctx.needs_input_grad[0]:
            dx = torch.empty((T, B, In), device=dev, dtype=torch.float32)
            for d in range(2):
                gemm(dpre.data_ptr() + 4 * G * d, 2 * G, 0, wi_il[d], In, 0, dx, In, M, In, G,
                     beta=0.0 if d == 0 else 1.0)
        P = ctx.params
        out = []
        if use16:
            tg = [_acc(P[i]) for i in (0, 4, 1, 5, 2, 3, 6, 7)]   # dW_ih f/r, dW_hh f/r, db_ih f, db_hh f, db_ih r, db_hh r

            def weight_grads():
                # dW_ih of both directions at once: [2G, In] = dpre16 [M, 2G]^T . xb16 [M, In]
                gemm_h16(dpre16, 2 * G, 1, xb16, Kp, 0, dwi_il2, In, 2 * G, In, M, a_bf16=True, b_bf16=True, beta=1.0)
                Mr = (T - 1) * B
                if T > 1:
                    # rows t=1.. of the forward direction pair with h[t-1]; rows ..T-2 of the reverse one with h[t+1]
                    gemm_h16(dpre16.data_ptr() + 2 * B * 2 * G, 2 * G, 1, hb16.data_ptr(), 2 * H, 0, dwh_il2[0], H, G, H,
                             Mr, a_bf16=True, b_bf16=True, beta=1.0)
                    gemm_h16(dpre16.data_ptr() + 2 * G, 2 * G, 1, hb16.data_ptr() + 2 * (B * 2 * H + H), 2 * H, 0,
                             dwh_il2[1], H, G, H, Mr, a_bf16=True, b_bf16=True, beta=1.0)
                # one pass: every gate-interleaved gradient of the layer accumulated into its nn.LSTM-order target
                call("deer_lstm_unprep", ptr(dwi_il2), ptr(dwh_il2), ptr(db_il), *[ptr(t[0]) for t in tg], H, In)

            if (dx is not None and _state["defer_wgrad"] and _state["direct_grad"] and _state.get("lstm_defer_wgrad", False)
                    and all(direct for _, direct in tg)):
                # (option, OFF: measured 3.755 vs 3.747 ms per step) trainer mode, a layer with an LSTM layer below it: its
                # three weight-gradient GEMMs (233 us at B = 256) leave the path from dx to the BPTT of the layer below and
                # run on the weight-gradient stream -- but CTA-pair GEMMs cannot share an SM with the recurrence, so they
                # only move behind that BPTT, where they meet the lower layer's own weight gradients
                cur = torch.cuda.current_stream()
                aux = _wgrad_stream()
                aux.wait_stream(cur)
                with torch.cuda.stream(aux):
                    weight_grads()
                for t_ in (dpre16, xb16, hb16, zbuf, db_il):
                    if t_ is not None:
                        t_.record_stream(aux)
                _wgrad["pending"] = True
            else:
                weight_grads()
            r = [None if direct else buf for buf, direct in tg]
            return dx, r[0], r[2], r[4], r[5], r[1], r[3], r[6], r[7], None, None, None, None, None, None
        for d in range(2):
            gp = dpre.data_ptr() + 4 * G * d
            dwi_il = torch.zeros((G, In), device=dev, dtype=torch.float32)
            dwh_il = torch.zeros((G, H), device=dev, dtype=torch.float32)
            Mr = (T - 1) * B
            gemm(gp, 2 * G, 1, x, In, 0, dwi_il, In, G, In, M, beta=1.0)
            if T > 1:
                if d == 0:   # rows t=1.. pair with h[t-1]
                    gemm(gp + 4 * B * 2 * G, 2 * G, 1, h.data_ptr(), 2 * H, 0, dwh_il, H, G, H, Mr, beta=1.0)
                else:        # rows t=..T-2 pair with h[t+1]
                    gemm(gp, 2 * G, 1, h.data_ptr() + 4 * (B * 2 * H + H), 2 * H, 0, dwh_il, H, G, H, Mr, beta=1.0)
            dwi, dwi_direct = _acc(P[4 * d])
            call("deer_gate_rows_interleave", ptr(dwi_il), ptr(dwi), H, In, 1, 1)
            dwh, dwh_direct = _acc(P[4 * d + 1])
            call("deer_gate_rows_interleave", ptr(dwh_il), ptr(dwh), H, H, 1, 1)
            dbs = []
            for pb in (P[4 * d + 2], P[4 * d + 3]):   # b_ih and b_hh receive the same gradient
                tgt, direct = _acc(pb)
                call("deer_gate_rows_interleave", ptr(db_il[d]), ptr(tgt), H, 1, 1, 1)
                dbs.append(None if direct else tgt)
            out.append((None if dwi_direct else dwi, None if dwh_direct else dwh, dbs[0], dbs[1]))
        (dwif, dwhf, dbif, dbhf), (dwir, dwhr, dbir, dbhr) = out
        return dx, dwif, dwhf, dbif, dbhf, dwir, dwhr, dbir, dbhr, None, None, None, None, None, None


def bilstm_layer(x_tm, wif, whf, bif, bhf, wir, whr, bir, bhr, input_dropout: float = 0.0, training: bool = False,
                 x_f16=None, emit_f16: bool = False, return_f16: bool = False, return_bf16: bool = False,
                 x_batch_major: bool = False, lengths=None):
    """engine AUTO/TF32: persistent cluster kernels when H == 256; SIMT: exact-fp32 stepwise; others: see lstm.cu.
    `lengths`: per-utterance lengths [B] on the device (sequence_lengths): nn.LSTM on
    pack_padded_sequence(x, lengths, batch_first=True, enforce_sorted=False); h is ~0 (<= 2^-83) at padded rows.  Cluster
    kernels on the 16-bit GEMM path only: the other engines raise DeerError.
    `x_batch_major`: x_tm is the batch_first [B,T,I] input of the first layer; on the cluster path its time-major 16-bit
    operand copies are written in one pass, elsewhere it is permuted first (ops.to_time_major).
    `input_dropout` (with `training`) applies nn.LSTM's inter-layer dropout to x_tm: fused into the layer's 16-bit
    operand casts on the cluster path, a separate kernel otherwise.
    `return_f16`: return (h, h_f16); with `emit_f16` h_f16 is the FP16 copy of h the recurrence kernel writes beside it
    (None when the path has none); pass it as `x_f16` to the next layer to skip that layer's operand cast (no-dropout
    case)."""
    cluster = _state["lstm_engine"] in (ENGINE_AUTO, ENGINE_TF32) and whf.shape[1] == 256
    if lengths is not None and not cluster:
        raise _lib.DeerError("deer_b200: LSTM lengths are built on the cluster kernels only (H == 256, engine AUTO)")
    drop = None
    bm = False
    if x_batch_major:
        bm = (cluster and _state["lstm_gemm16"] and _state["engine"] == ENGINE_AUTO and _state.get("lstm_bm_input", True)
              and not (training and input_dropout > 0.0) and not (x_tm.requires_grad and torch.is_grad_enabled()))
        if not bm:
            x_tm = to_time_major(x_tm)
    if training and input_dropout > 0.0:
        fusable = (cluster and _state["fuse_lstm_dropout"] and _state["lstm_gemm16"] and
                   _state["engine"] == ENGINE_AUTO and x_tm.shape[-1] % 8 == 0)
        if fusable:
            off = _dropout_state["offset"]
            _dropout_state["offset"] = off + (x_tm.numel() + 3) // 4
            drop = (float(input_dropout), _dropout_seed(), off)
        else:
            x_tm = dropout(x_tm, input_dropout, True)
    if cluster:
        want = bool(emit_f16 and _state["lstm_gemm16"] and _state["engine"] == ENGINE_AUTO)
        # (a custom Function's forward always runs with grad mode off: the caller's mode is passed in, so that an
        # inference forward keeps nothing for BPTT and can use the no-keep kernels)
        h, h16, hb16 = _BiLSTMLayerCluster.apply(x_tm, wif, whf, bif, bhf, wir, whr, bir, bhr, drop,
                                                 x_f16 if drop is None else None, want, torch.is_grad_enabled(), bm,
                                                 lengths)
        if return_bf16:     # (h, FP16 copy or None, BF16 copy or None): the 16-bit shadows the recurrence kernel wrote
            return h, (h16 if h16.numel() else None), (hb16 if hb16.numel() else None)
        return (h, h16 if h16.numel() else None) if return_f16 else h
    h = _BiLSTMLayer.apply(x_tm, wif, whf, bif, bhf, wir, whr, bir, bhr, torch.is_grad_enabled())
    if return_bf16:
        return h, None, None
    return (h, None) if return_f16 else h


# ----------------------------------------------------------------------------------------------- Conv1d(k=3) + BN
class _Conv1dK3(torch.autograd.Function):
    """nn.Conv1d(Cin,Cout,3,padding=1) on channels-last x [B,T,Cin] -> [B,T,Cout]; w [Cout,Cin,3].  lengths (device [B]):
    each clip x[b, :L_b] is convolved alone -- x is masked to zero rows at t >= L_b before the im2col, and dx after the
    col2im (0 at padded frames)."""

    @staticmethod
    def forward(ctx, x, w, b, lengths=None):
        x = _req(x, "x").contiguous()
        B, T, Cin = x.shape
        Cout = w.shape[0]
        if lengths is not None:
            x = _mask_padding(x, lengths)
        col = torch.empty((B * T, 3 * Cin), device=x.device, dtype=torch.float32)
        call("deer_im2col3", ptr(x), ptr(col), B, T, Cin)
        wk = torch.empty((Cout, 3 * Cin), device=x.device, dtype=torch.float32)
        call("deer_conv3_weight_pack", ptr(w.contiguous()), ptr(wk), Cout, Cin, 0)
        y = torch.empty((B, T, Cout), device=x.device, dtype=torch.float32)
        ce = _state["conv_exact"]
        # small problems (the im2col path): forward taps on the fp32-grade engine, like every other forward contraction
        exact_fwd = (ce & 1) or (_state["split_fwd"] and _state["engine"] == ENGINE_AUTO)
        gemm(col, 3 * Cin, 0, wk, 3 * Cin, 1, y, Cout, B * T, Cout, 3 * Cin, bias=b,
             engine=_state["exact_engine"] if exact_fwd else None)
        ctx.save_for_backward(col, wk)
        ctx.dims = (B, T, Cin, Cout)
        ctx.params = (w, b)
        ctx.lengths = lengths
        return y

    @staticmethod
    def backward(ctx, dy):
        col, wk = ctx.saved_tensors
        B, T, Cin, Cout = ctx.dims
        dy = dy.contiguous()
        M = B * T
        dx = None
        if ctx.needs_input_grad[0]:
            dcol = torch.empty_like(col)
            gemm(dy, Cout, 0, wk, 3 * Cin, 0, dcol, 3 * Cin, M, 3 * Cin, Cout,
                 engine=_state["exact_engine"] if (_state["conv_exact"] & 2) else None)
            dx = torch.empty((B, T, Cin), device=dy.device, dtype=torch.float32)
            call("deer_col2im3", ptr(dcol), ptr(dx), B, T, Cin)
            if ctx.lengths is not None:
                dx = _mask_padding(dx, ctx.lengths)
        dwk = zeros_scratch(tuple(wk.shape), dy.device)
        gemm(dy, Cout, 1, col, 3 * Cin, 0, dwk, 3 * Cin, Cout, 3 * Cin, M, beta=1.0,
             engine=_state["exact_engine"] if (_state["conv_exact"] & 2) else None)
        dw, dw_direct = _acc(ctx.params[0])
        call("deer_conv3_weight_pack", ptr(dwk), ptr(dw), Cout, Cin, 1)
        db, db_direct = _acc(ctx.params[1])
        call("deer_bias_act_bwd", ptr(dy), Cout, None, 0, None, 0, ptr(db), M, Cout, 0)
        return dx, None if dw_direct else dw, None if db_direct else db, None


class _Conv1dK3Window(torch.autograd.Function):
    """The same convolution without an im2col matrix: x is copied once into a zero-row-padded layout xp
    ([1 zero row][sample: T rows][zero row]...), whose OVERLAPPING row windows xp[q:q+3] (3*Cin contiguous floats, row
    pitch Cin) are exactly the im2col rows.  The TMA engine reads those windows straight from xp (a tensor map whose row
    pitch is smaller than its row length): forward y_big = windows . wk^T, backward dwk = dy_big^T . windows and
    dx_p += dy_big . wk accumulated into overlapping rows by the TMA reduce-add epilogue (no dcol, no col2im).
    Rows centred on a pad row are garbage in y_big and are dropped by the un-padding copy; dy_big has zeros there."""

    @staticmethod
    def forward(ctx, x, w, b, drop=None, lengths=None):
        """drop = (p, seed, offset, step tensor or None): the nn.Dropout in front of the convolution (encoders.py:453-454)
        folded into the padding pass (forward) and the un-padding pass (backward): same Philox stream as ops.dropout.
        lengths (device [B]): frames t >= L_b are pad rows of xp as well (zeros, not read), and the un-padding pass of
        the backward writes dx = 0 there."""
        x = _req(x, "x").contiguous()
        B, T, Cin = x.shape
        Cout = w.shape[0]
        dev = x.device
        Mp = B * (T + 1)                                        # window rows (one per padded row centre)
        xp = torch.empty((Mp + 2, Cin), device=dev, dtype=torch.float32)
        split = _split_fwd_ok(Mp, Cout, 3 * Cin) and Cin % 8 == 0
        dp, dseed, doff, dstep = drop if drop is not None else (0.0, 0, 0, None)
        xh = xl = None
        if split:   # the hi / lo FP16 copies of the padded rows keep the overlapping-window geometry (row pitch Cin)
            xh = torch.empty((Mp + 2, Cin), device=dev, dtype=torch.float16)
            xl = torch.empty((Mp + 2, Cin), device=dev, dtype=torch.float16)
        # one pass: dropout, zero pad rows, fp32 copy (weight gradient) and the split-precision A operand
        _rows_pad_fused(x, xp, xh, xl, lengths, B, T, Cin, 0, float(dp), int(dseed), int(doff), dstep)
        wk = torch.empty((Cout, 3 * Cin), device=dev, dtype=torch.float32)
        call("deer_conv3_weight_pack", ptr(w.contiguous()), ptr(wk), Cout, Cin, 0)
        y_big = torch.empty((Mp, Cout), device=dev, dtype=torch.float32)
        if split:
            wh, wl, _ = cast_split16(wk)
            gemm_split(xh, xl, Cin, wh, wl, 3 * Cin, y_big, Cout, Mp, Cout, 3 * Cin, bias=b)   # lda = Cin < K = 3 Cin
        else:
            gemm(xp, Cin, 0, wk, 3 * Cin, 1, y_big, Cout, Mp, Cout, 3 * Cin, bias=b)      # lda = Cin < K = 3 Cin
        y = torch.empty((B, T, Cout), device=dev, dtype=torch.float32)
        call("deer_rows_pad", ptr(y_big), ptr(y), B, T, Cout, 0, 0, 1)
        ctx.save_for_backward(xp, wk)
        ctx.dims = (B, T, Cin, Cout)
        ctx.params = (w, b)
        ctx.drop = (float(dp), int(dseed), int(doff), dstep)
        ctx.lengths = lengths
        return y

    @staticmethod
    def backward(ctx, dy):
        xp, wk = ctx.saved_tensors
        B, T, Cin, Cout = ctx.dims
        dev = dy.device
        dy = dy.contiguous()
        Mp = B * (T + 1)
        dy_big = torch.empty((Mp, Cout), device=dev, dtype=torch.float32)
        db, db_direct = _acc(ctx.params[1])
        # one pass over dy: the padded copy (zero rows at the pad centres) and the bias gradient's column sums
        call("deer_rows_pad_colsum", ptr(dy), ptr(dy_big), ptr(db), B, T, Cout)
        dx = None
        bf = _bwd16_ok(Mp) and Cin % 8 == 0 and Cout % 8 == 0
        if bf:   # BF16 operands on the 16-bit tcgen05 engine (same overlapping-row geometry)
            dyb = cast16(dy_big, bf16=True)
            xpb = cast16(xp, bf16=True)
        if ctx.needs_input_grad[0]:
            dx_p = zeros_scratch((Mp + 2, Cin), dev)
            if bf:
                wkb = cast16(wk, bf16=True)
                gemm_h16(dyb, Cout, 0, wkb, 3 * Cin, 0, dx_p, Cin, Mp, 3 * Cin, Cout, a_bf16=True, b_bf16=True, beta=1.0)
            else:
                gemm(dy_big, Cout, 0, wk, 3 * Cin, 0, dx_p, Cin, Mp, 3 * Cin, Cout, beta=1.0)   # ldc = Cin < N: overlapped
            dx = torch.empty((B, T, Cin), device=dev, dtype=torch.float32)
            dp, dseed, doff, dstep = ctx.drop
            _rows_pad_fused(dx_p, dx, None, None, ctx.lengths, B, T, Cin, 1, dp, dseed, doff, dstep)
        dwk = zeros_scratch(tuple(wk.shape), dev)
        if bf:
            gemm_h16(dyb, Cout, 1, xpb, Cin, 0, dwk, 3 * Cin, Cout, 3 * Cin, Mp, a_bf16=True, b_bf16=True, beta=1.0)
        else:
            gemm(dy_big, Cout, 1, xp, Cin, 0, dwk, 3 * Cin, Cout, 3 * Cin, Mp, beta=1.0)         # ldb = Cin < N = 3 Cin
        dw, dw_direct = _acc(ctx.params[0])
        call("deer_conv3_weight_pack", ptr(dwk), ptr(dw), Cout, Cin, 1)
        return dx, None if dw_direct else dw, None if db_direct else db, None, None


def _rows_pad_fused(src, dst, hi, lo, lengths, B, T, C, direction, dp, dseed, doff, dstep):
    """The sliding-window convolution's padding (direction 0) / un-padding (1) pass, lead = tail = 1 row; with lengths
    the frames t >= L_b are pad rows too."""
    hp = None if hi is None else hi.data_ptr()
    lp = None if lo is None else lo.data_ptr()
    if lengths is not None:
        call("deer_rows_pad_fused_len", ptr(src), ptr(dst), hp, lp, lengths.data_ptr(), _len_i64(lengths), B, T, C, 1, 1,
             direction, dp, dseed, doff, ptr(dstep))
    else:
        call("deer_rows_pad_fused", ptr(src), ptr(dst), hp, lp, B, T, C, 1, 1, direction, dp, dseed, doff, ptr(dstep))


def set_conv_window(on: bool):
    """Conv1d(k=3) through the sliding-window (overlapping-row TMA) path (default) or through an im2col matrix."""
    _state["conv_window"] = bool(on)


def conv1d_k3(x, w, b, dropout_p: float = 0.0, training: bool = False, lengths=None):
    """Conv1d(k=3, padding=1) of dropout(x) (dropout_p > 0 and training: the nn.Dropout in front of the convolution,
    encoders.py:453-454).  Large batches on the TMA engine use the sliding-window path (no im2col matrix; the dropout
    rides on its padding / un-padding passes); small ones (the CTA-pair kernel needs > 256 rows), forced engines and odd
    channel counts keep the im2col + GEMM path behind a separate dropout node.  Both draw the same masks.
    `lengths` [B] (see sequence_lengths): sample b is the clip x[b, :L_b], convolved with zero padding at both of ITS
    ends (the tap at t = L_b reads 0); the output rows t >= L_b are finite but meaningless, and the input gradient is
    exactly 0 there."""
    B, T, Cin = x.shape
    Cout = w.shape[0]
    lengths = sequence_lengths(lengths, B, T, x.device)
    dropping = training and dropout_p > 0.0
    if (_state.get("conv_window", True) and not _state["conv_exact"] and _state["engine"] == ENGINE_AUTO and
            B * (T + 1) > 256 and Cin % 4 == 0 and
            Cout % 4 == 0 and Cin >= 32 and Cout > 256):   # dW runs with M = Cout rows on the CTA-pair kernel
        drop = None
        if dropping and _state.get("conv_drop_fused", True):
            off = _dropout_state["offset"]
            _dropout_state["offset"] = off + (x.numel() + 3) // 4
            drop = (float(dropout_p), _dropout_seed(), off, _dropout_state["step"])
        elif dropping:
            x = dropout(x, dropout_p, training)
        return _Conv1dK3Window.apply(x, w, b, drop, lengths)
    if dropping:
        x = dropout(x, dropout_p, training)
    return _Conv1dK3.apply(x, w, b, lengths)


def set_conv_dropout_fused(on: bool):
    """Dropout in front of a sliding-window Conv1d inside its padding passes (default) or as a separate node (ablation /
    the reference point of the equality test)."""
    _state["conv_drop_fused"] = bool(on)


class _BNReLU(torch.autograd.Function):
    """nn.BatchNorm1d (channels-last rows) followed by ReLU.  lengths (device [B], x [B,T,C]): the rows are the valid
    frames t < L_b only -- nn.BatchNorm1d on those packed into one [N, C] batch, N = sum_b L_b counted on the device
    (stats [2C+1]: mean, biased var, N); y = 0 and dx = 0 at padded rows."""

    @staticmethod
    def forward(ctx, x, g, b, running_mean, running_var, nbt, training, momentum, eps, lengths=None):
        x = _req(x, "x").contiguous()
        C = x.shape[-1]
        M = x.numel() // C
        y = torch.empty_like(x)
        nbt_p = None if nbt is None else nbt.data_ptr()
        if lengths is not None:
            B, T = x.shape[0], x.shape[1]
            lp, li = lengths.data_ptr(), _len_i64(lengths)
        if training:
            if lengths is not None:
                stats = torch.empty(2 * C + 1, device=x.device, dtype=torch.float32)
                call("deer_bn_stats_len", ptr(x), ptr(stats), lp, li, B, T, C)
                call("deer_bn_update_running_len", ptr(stats), ptr(running_mean), ptr(running_var), nbt_p, C,
                     float(momentum))
                mean, var = stats[:C], stats[C:2 * C]     # views: the backward reads N at mean[2C]
            else:
                stats = torch.empty((2, C), device=x.device, dtype=torch.float32)
                call("deer_bn_stats", ptr(x), ptr(stats), M, C)
                call("deer_bn_update_running", ptr(stats), ptr(running_mean), ptr(running_var), nbt_p, M, C,
                     float(momentum))
                mean, var = stats[0], stats[1]
        else:
            mean, var = running_mean, running_var
        if lengths is not None:
            call("deer_bn_relu_fwd_len", ptr(x), ptr(mean), ptr(var), ptr(g), ptr(b), ptr(y), lp, li, B, T, C,
                 float(eps))
        else:
            call("deer_bn_relu_fwd", ptr(x), ptr(mean), ptr(var), ptr(g), ptr(b), ptr(y), M, C, float(eps))
        ctx.save_for_backward(x, y, mean.clone() if not training else mean, var.clone() if not training else var, g)
        ctx.cfg = (M, C, float(eps), bool(training))
        ctx.params = (g, b)
        ctx.lengths = lengths
        return y

    @staticmethod
    def backward(ctx, dy):
        x, y, mean, var, g = ctx.saved_tensors
        M, C, eps, training = ctx.cfg
        dy = dy.contiguous()
        dx = torch.empty_like(x)
        dg, dg_direct = _acc(ctx.params[0])
        db, db_direct = _acc(ctx.params[1])
        scratch = torch.empty((2, C), device=x.device, dtype=torch.float32)
        lengths = ctx.lengths
        if lengths is not None:
            call("deer_bn_relu_bwd_len", ptr(dy), ptr(x), ptr(y), ptr(mean), ptr(var), ptr(g), ptr(dx), ptr(dg),
                 ptr(db), ptr(scratch), lengths.data_ptr(), _len_i64(lengths), x.shape[0], x.shape[1], C, eps,
                 int(training))
        else:
            call("deer_bn_relu_bwd", ptr(dy), ptr(x), ptr(y), ptr(mean), ptr(var), ptr(g), ptr(dx), ptr(dg), ptr(db),
                 ptr(scratch), M, C, eps, int(training))
        return dx, None if dg_direct else dg, None if db_direct else db, None, None, None, None, None, None, None


def batchnorm_relu(x, g, b, running_mean, running_var, nbt, training, momentum=0.1, eps=1e-5, lengths=None):
    """`lengths` [B] (see sequence_lengths) with x [B,T,C]: the statistics, the output and the gradients cover the frames
    t < L_b only; padded rows of y and dx are exactly 0 and their content in x does not matter."""
    if lengths is not None:
        if x.dim() != 3:
            raise _lib.DeerError(f"deer_b200: batchnorm_relu with lengths needs x [B,T,C], got {tuple(x.shape)}")
        lengths = sequence_lengths(lengths, x.shape[0], x.shape[1], x.device)
    return _BNReLU.apply(x, g, b, running_mean, running_var, nbt, training, momentum, eps, lengths)


# ----------------------------------------------------------------------------------------------- 2-token MHA core
class _MHA2(torch.autograd.Function):
    """qkv [B,2,3E] (packed q|k|v per token) -> (token-mean context [B,E], head-averaged weights [B,2,2])."""

    @staticmethod
    def forward(ctx, qkv, heads):
        qkv = _req(qkv, "qkv").contiguous()
        B, two, E3 = qkv.shape
        assert two == 2
        E = E3 // 3
        cmean = torch.empty((B, E), device=qkv.device, dtype=torch.float32)
        attw = torch.empty((B, 2, 2), device=qkv.device, dtype=torch.float32)
        probs = torch.empty((B, heads, 2, 2), device=qkv.device, dtype=torch.float32)
        call("deer_mha2_fwd", ptr(qkv), None, ptr(cmean), ptr(attw), ptr(probs), B, E, heads)
        ctx.save_for_backward(qkv, probs)
        ctx.heads = heads
        # the attention weights are a reporting output (no loss term reads them): without this autograd hands backward a
        # zero-filled [B,2,2] tensor for them -- one at::fill launch inside the serial fusion chain of every step
        ctx.set_materialize_grads(False)
        return cmean, attw

    @staticmethod
    def backward(ctx, dcmean, dattw):
        qkv, probs = ctx.saved_tensors
        B, _, E3 = qkv.shape
        if dcmean is None:
            dcmean = zeros_scratch((B, E3 // 3), qkv.device)
        dqkv = torch.empty_like(qkv)
        call("deer_mha2_bwd", None, ptr(dcmean.contiguous()), ptr(dattw.contiguous()) if dattw is not None else None,
             ptr(qkv), ptr(probs), ptr(dqkv), B, E3 // 3, ctx.heads)
        return dqkv, None


def mha2_core(qkv, heads):
    return _MHA2.apply(qkv, heads)


# ----------------------------------------------------------------------------------------------- grouped Linear
def _uniform_stride(ptrs):
    """Element stride between consecutive fp32 pointers if it is the same for all of them (None otherwise)."""
    if len(ptrs) < 2:
        return None
    d = ptrs[1] - ptrs[0]
    if d % 16 != 0 or any(ptrs[i + 1] - ptrs[i] != d for i in range(len(ptrs) - 1)):
        return None
    return d // 4


class _GroupedLinear(torch.autograd.Function):
    """out[:, g, :] = act(x_g W_g^T + b_g) for g in range(G); out [M,G,N].  Inputs may be strided row views
    (e.g. slices out[:, g, :] of a previous grouped output), so chains of per-head layers need no copies."""

    @staticmethod
    def forward(ctx, act, G, *args):
        ws, bs, xs = args[:G], args[G:2 * G], args[2 * G:]
        N = ws[0].shape[0]
        rows = [_rows2d(_req(x, "input")) for x in xs]
        M = rows[0][1]
        out = torch.empty((M, G, N), device=ws[0].device, dtype=torch.float32)
        # One batched launch when the groups' operands are evenly spaced in memory (the per-head layers of the NIG head:
        # equal-sized heads laid out back to back in the trainer's flat parameter buffer; inputs either one shared
        # tensor or slices of a previous grouped output)
        same = (all(r[2] == rows[0][2] and r[3] == rows[0][3] for r in rows) and
                all(w.shape == ws[0].shape and w.stride(0) == ws[0].stride(0) for w in ws) and
                all(b is not None for b in bs))
        sx = sw = sb = None
        if same and G > 1 and _state["grouped_batched"]:
            xp = [r[0].data_ptr() for r in rows]
            sx = 0 if all(q == xp[0] for q in xp) else _uniform_stride(xp)
            sw = _uniform_stride([w.data_ptr() for w in ws])
            sb = _uniform_stride([b.data_ptr() for b in bs])
        batched = sx is not None and sw is not None and sb is not None
        if batched:
            x2, _, K, ld = rows[0]
            gemm(x2, ld, 0, ws[0], ws[0].stride(0), 1, out, G * N, M, N, K, bias=bs[0], act=act, batch=G, sA=sx, sB=sw,
                 sC=N, sBias=sb, engine=_fwd_engine(M, True))
        else:
            for g in range(G):
                x2, _, K, ld = rows[g]
                gemm(x2, ld, 0, ws[g], ws[g].stride(0), 1, out.data_ptr() + 4 * g * N, G * N, M, N, K, bias=bs[g],
                     act=act, engine=_fwd_engine(M, True))
        ctx.batched = (sx, sw) if batched else None
        ctx.act, ctx.G = act, G
        ctx.params = (ws, bs)
        ctx.meta = [(r[3], r[2]) for r in rows]
        ctx.in_shapes = [x.shape for x in xs]
        ctx.save_for_backward(out if act != 0 else None, *ws, *[r[0] for r in rows])
        return out

    @staticmethod
    def backward(ctx, dout):
        G, act = ctx.G, ctx.act
        saved = ctx.saved_tensors
        out, ws, xs = saved[0], saved[1:1 + G], saved[1 + G:]
        dout = dout.contiguous()
        M, _, N = dout.shape
        dev = dout.device
        pws, pbs = ctx.params
        db_acc = [_acc(pbs[g]) if ctx.needs_input_grad[2 + G + g] else (None, False) for g in range(G)]
        dbs = [a[0] for a in db_acc]
        dz = torch.empty_like(dout) if act != 0 else dout
        for g in range(G):
            off = 4 * g * N
            if act != 0:
                call("deer_bias_act_bwd", dout.data_ptr() + off, G * N, out.data_ptr() + off, G * N,
                     dz.data_ptr() + off, G * N, ptr(dbs[g]), M, N, act)
            elif dbs[g] is not None:
                call("deer_bias_act_bwd", dout.data_ptr() + off, G * N, None, 0, None, 0, ptr(dbs[g]), M, N, 0)
        dws, dxs = [], []
        if ctx.batched is not None and all(ctx.needs_input_grad[2 + g] for g in range(G)):
            # batched weight gradients (and input gradients when the groups have distinct inputs): one launch each
            sx, sw = ctx.batched
            ld, K = ctx.meta[0]
            dw_acc = [_acc(pws[g]) for g in range(G)]
            sdw = _uniform_stride([a[0].data_ptr() for a in dw_acc])
            need_dx = [ctx.needs_input_grad[2 + 2 * G + g] for g in range(G)]
            # (sdw == 0: one weight shared by the groups, e.g. the packed in_proj of the two-token attention -- its
            # gradient contributions must be accumulated one after the other, not by concurrent batch entries)
            if sdw and (sx != 0 or not any(need_dx)) and (all(need_dx) or not any(need_dx)):
                gemm(dz, G * N, 1, xs[0], ld, 0, dw_acc[0][0], K, N, K, M, beta=1.0, batch=G, sA=N, sB=sx, sC=sdw,
                     engine=_bwd_engine(M, True))
                dws = [None if direct else buf for buf, direct in dw_acc]
                if all(need_dx):
                    dxa = torch.empty((G, M, K), device=dev, dtype=torch.float32)
                    gemm(dz, G * N, 0, ws[0], ws[0].stride(0), 0, dxa, K, M, K, N, batch=G, sA=N, sB=sw, sC=M * K,
                         engine=_bwd_engine(M, True))
                    dxs = [dxa[g].view(ctx.in_shapes[g]) for g in range(G)]
                else:
                    dxs = [None] * G
                dbs = [None if a[1] else a[0] for a in db_acc]
                return (None, None, *dws, *dbs, *dxs)
        for g in range(G):
            ld, K = ctx.meta[g]
            zp = dz.data_ptr() + 4 * g * N
            if ctx.needs_input_grad[2 + g]:
                dw, direct = _acc(pws[g])
                gemm(zp, G * N, 1, xs[g], ld, 0, dw, K, N, K, M, beta=1.0, engine=_bwd_engine(M, True))
                dws.append(None if direct else dw)
            else:
                dws.append(None)
            if ctx.needs_input_grad[2 + 2 * G + g]:
                dx = torch.empty((M, K), device=dev, dtype=torch.float32)
                gemm(zp, G * N, 0, ws[g], ws[g].stride(0), 0, dx, K, M, K, N, engine=_bwd_engine(M, True))
                dxs.append(dx.view(ctx.in_shapes[g]))
            else:
                dxs.append(None)
        dbs = [None if a[1] else a[0] for a in db_acc]
        return (None, None, *dws, *dbs, *dxs)


class _GroupedLinearX3(torch.autograd.Function):
    """out[:, g, :] = dropout(act(x_g W_g^T + b_g)), out [M,G,N], on the fused 3xTF32 engine: one batched launch when the
    groups' operands are evenly spaced (per-head layers laid out back to back in the trainer's flat buffers), one launch
    per group otherwise.  Backward: gate (activation / dropout derivative from the saved output) and bias gradients
    inside the GEMMs; groups that share one input accumulate ONE input gradient (no per-group temporaries + adds)."""

    @staticmethod
    def forward(ctx, act, drop, G, sliced, *args):
        ws, bs, xs = args[:G], args[G:2 * G], args[2 * G:]
        N = ws[0].shape[0]
        if sliced:      # ONE input [M,G,K]: group g reads x[:, g] (its gradient comes back as one [M,G,K] tensor)
            x3 = _req(xs[0], "input").contiguous()
            ctx.sliced_shape = x3.shape
            xs = [x3[:, g] for g in range(G)]
        ctx.sliced = bool(sliced)
        rows = [_rows2d(_req(x, "input")) for x in xs]
        M = rows[0][1]
        out = torch.empty((M, G, N), device=ws[0].device, dtype=torch.float32)
        same = (all(r[2] == rows[0][2] and r[3] == rows[0][3] for r in rows) and
                all(w.shape == ws[0].shape and w.stride(0) == ws[0].stride(0) for w in ws) and
                all(b is not None for b in bs))
        sx = sw = sb = None
        if same and G > 1 and _state["grouped_batched"]:
            xp = [r[0].data_ptr() for r in rows]
            sx = 0 if all(q == xp[0] for q in xp) else _uniform_stride(xp)
            wp = [w.data_ptr() for w in ws]
            sw = 0 if all(q == wp[0] for q in wp) else _uniform_stride(wp)
            bp = [b.data_ptr() for b in bs]
            sb = 0 if all(q == bp[0] for q in bp) else _uniform_stride(bp)
        batched = sx is not None and sw is not None and sb is not None
        if batched:
            x2, _, K, ld = rows[0]
            gemm_x3(x2, ld, 0, ws[0], ws[0].stride(0), 1, out, G * N, M, N, K, bias=bs[0], act=act, batch=G, sA=sx, sB=sw,
                    sC=N, sBias=sb, drop=drop, drop_ld=G * N, drop_batch_stride=N)
        else:
            for g in range(G):
                x2, _, K, ld = rows[g]
                gemm_x3(x2, ld, 0, ws[g], ws[g].stride(0), 1, out.data_ptr() + 4 * g * N, G * N, M, N, K, bias=bs[g],
                        act=act, drop=drop, drop_ld=G * N, drop_col0=g * N)
        ctx.batched = (sx, sw) if batched else None
        ctx.act, ctx.G = act, G
        ctx.drop_p = drop[0] if drop is not None else 0.0
        ctx.params = (ws, bs)
        ctx.meta = [(r[3], r[2]) for r in rows]
        ctx.in_shapes = [x.shape for x in xs]
        ctx.save_for_backward(out if (act != 0 or ctx.drop_p > 0.0) else None, *ws, *[r[0] for r in rows])
        return out

    @staticmethod
    def backward(ctx, dout):
        G, act = ctx.G, ctx.act
        saved = ctx.saved_tensors
        out, ws, xs = saved[0], saved[1:1 + G], saved[1 + G:]
        dout = dout.contiguous()
        M, _, N = dout.shape
        dev = dout.device
        pws, pbs = ctx.params
        gmode = _GATE_MODE[act] if out is not None else 0
        gscale = 1.0 / (1.0 - ctx.drop_p) if ctx.drop_p > 0.0 else 1.0
        LD = G * N
        need_w = [ctx.needs_input_grad[4 + g] for g in range(G)]
        need_b = [ctx.needs_input_grad[4 + G + g] for g in range(G)]
        need_x = [ctx.needs_input_grad[4 + 2 * G + (0 if ctx.sliced else g)] for g in range(G)]
        # ---- weight (+ bias) gradients
        dws, dbs = [None] * G, [None] * G
        w_acc = [_acc(pws[g]) if need_w[g] else (None, False) for g in range(G)]
        b_acc = [_acc(pbs[g]) if need_b[g] else (None, False) for g in range(G)]
        shared_w = all(w.data_ptr() == ws[0].data_ptr() for w in ws)   # one weight used by every group (packed in_proj)
        if shared_w and G > 1:
            # the contributions of the groups accumulate into ONE gradient buffer, one after the other
            w_acc = [w_acc[0]] * G
            b_acc = [b_acc[0]] * G
        done_batched = False
        if ctx.batched is not None and all(need_w) and all(need_b) and not shared_w:
            sx, sw = ctx.batched
            ld, K = ctx.meta[0]
            sdw = _uniform_stride([a[0].data_ptr() for a in w_acc])
            sdb = _uniform_stride([a[0].data_ptr() for a in b_acc])
            if sdw and sdb:
                gemm_x3(dout, LD, 1, xs[0], ld, 0, w_acc[0][0], K, N, K, M, beta=1.0, batch=G, sA=N, sB=sx, sC=sdw,
                        gate=out, ldgate=LD, gate_mode=gmode, gate_scale=gscale, sGate=N, colsum=b_acc[0][0],
                        sColsum=sdb)
                done_batched = True
        if not done_batched:
            for g in range(G):
                if not need_w[g]:
                    continue
                ld, K = ctx.meta[g]
                off = 4 * g * N
                gemm_x3(dout.data_ptr() + off, LD, 1, xs[g], ld, 0, w_acc[g][0], K, N, K, M, beta=1.0,
                        gate=None if out is None else out.data_ptr() + off, ldgate=LD, gate_mode=gmode,
                        gate_scale=gscale, colsum=b_acc[g][0] if need_b[g] else None)
        for g in range(G):
            if shared_w and g > 0:
                continue
            dws[g] = None if (w_acc[g][0] is None or w_acc[g][1]) else w_acc[g][0]
            dbs[g] = None if (b_acc[g][0] is None or b_acc[g][1]) else b_acc[g][0]
        # ---- input gradients
        dxs = [None] * G
        shared_x = G > 1 and all(x.data_ptr() == xs[0].data_ptr() for x in xs) and all(m == ctx.meta[0] for m in ctx.meta)
        if ctx.sliced:
            dx_full = None
            if need_x[0]:
                K = ctx.meta[0][1]
                dx_full = torch.empty((M, G, K), device=dev, dtype=torch.float32)
                swp = _uniform_stride([w.data_ptr() for w in ws]) if not shared_w else 0
                if swp is not None and all(w.stride(0) == ws[0].stride(0) for w in ws):
                    gemm_x3(dout, LD, 0, ws[0], ws[0].stride(0), 0, dx_full, G * K, M, K, N, batch=G, sA=N, sB=swp, sC=K,
                            gate=out, ldgate=LD, gate_mode=gmode, gate_scale=gscale, sGate=N)
                else:
                    for g in range(G):
                        off = 4 * g * N
                        gemm_x3(dout.data_ptr() + off, LD, 0, ws[g], ws[g].stride(0), 0, dx_full.data_ptr() + 4 * g * K,
                                G * K, M, K, N, gate=None if out is None else out.data_ptr() + off, ldgate=LD,
                                gate_mode=gmode, gate_scale=gscale)
            return (None, None, None, None, *dws, *dbs, dx_full)
        if any(need_x):
            if shared_x:
                # one input feeds every group: dx = sum_g dz_g W_g -- a single contraction over K = G*N when the weights
                # are stacked back to back, otherwise accumulated group by group into the same buffer
                ld, K = ctx.meta[0]
                dx = torch.empty((M, K), device=dev, dtype=torch.float32)
                swp = _uniform_stride([w.data_ptr() for w in ws])
                if swp == N * ws[0].stride(0) and all(w.stride(0) == ws[0].stride(0) for w in ws):
                    gemm_x3(dout, LD, 0, ws[0], ws[0].stride(0), 0, dx, K, M, K, G * N, gate=out, ldgate=LD,
                            gate_mode=gmode, gate_scale=gscale)
                else:
                    for g in range(G):
                        off = 4 * g * N
                        gemm_x3(dout.data_ptr() + off, LD, 0, ws[g], ws[g].stride(0), 0, dx, K, M, K, N,
                                beta=0.0 if g == 0 else 1.0, gate=None if out is None else out.data_ptr() + off,
                                ldgate=LD, gate_mode=gmode, gate_scale=gscale)
                dxs[0] = dx.view(ctx.in_shapes[0])
            elif ctx.batched is not None and all(need_x):
                sx, sw = ctx.batched
                ld, K = ctx.meta[0]
                dxa = torch.empty((G, M, K), device=dev, dtype=torch.float32)
                gemm_x3(dout, LD, 0, ws[0], ws[0].stride(0), 0, dxa, K, M, K, N, batch=G, sA=N, sB=sw, sC=M * K, gate=out,
                        ldgate=LD, gate_mode=gmode, gate_scale=gscale, sGate=N)
                dxs = [dxa[g].view(ctx.in_shapes[g]) for g in range(G)]
            else:
                for g in range(G):
                    if not need_x[g]:
                        continue
                    ld, K = ctx.meta[g]
                    off = 4 * g * N
                    dx = torch.empty((M, K), device=dev, dtype=torch.float32)
                    gemm_x3(dout.data_ptr() + off, LD, 0, ws[g], ws[g].stride(0), 0, dx, K, M, K, N,
                            gate=None if out is None else out.data_ptr() + off, ldgate=LD, gate_mode=gmode,
                            gate_scale=gscale)
                    dxs[g] = dx.view(ctx.in_shapes[g])
        return (None, None, None, None, *dws, *dbs, *dxs)


def grouped_linear(xs: Sequence[torch.Tensor], ws: Sequence[torch.Tensor], bs: Sequence[torch.Tensor], act="none",
                   dropout: float = 0.0, training: bool = False):
    """Per-group nn.Linear (+ activation) (+ nn.Dropout) into one [M,G,N] buffer (the D heads of the NIG head; the packed
    q|k|v projection of the two fusion tokens)."""
    G = len(ws)
    a = ACT[act]
    sliced = isinstance(xs, torch.Tensor)      # one [M,G,K] tensor: group g reads xs[:, g]
    if _fused_chain() and all(b is not None for b in bs) and (dropout <= 0.0 or not training or a == 1):
        M = xs.shape[0] if sliced else xs[0].numel() // xs[0].shape[-1]
        drop = _take_dropout(M * G * ws[0].shape[0], dropout, training)
        return _GroupedLinearX3.apply(a, drop, G, sliced, *ws, *bs, *([xs] if sliced else xs))
    if sliced:
        xs = [xs[:, g] for g in range(G)]
    return _apply_dropout(_GroupedLinear.apply(a, G, *ws, *bs, *xs), dropout, training)


# ----------------------------------------------------------------------------------------------- NIG head + losses
class _NigHead(torch.autograd.Function):
    """evidence [...,4] -> stacked [7, ...] = (mu, nu, alpha, beta, aleatoric, epistemic, total)."""

    @staticmethod
    def forward(ctx, evidence):
        e = _req(evidence, "evidence").contiguous()
        n = e.numel() // 4
        out = torch.empty((7, n), device=e.device, dtype=torch.float32)
        p = [out[i].data_ptr() for i in range(7)]
        call("deer_nig_head_fwd", ptr(e), *p, n)
        ctx.save_for_backward(e)
        return out.view(7, *e.shape[:-1])

    @staticmethod
    def backward(ctx, dout):
        (e,) = ctx.saved_tensors
        n = e.numel() // 4
        d = dout.contiguous().view(7, n)
        de = torch.empty_like(e)
        call("deer_nig_head_bwd", ptr(e), *[d[i].data_ptr() for i in range(7)], ptr(de), n)
        return de


def nig_head(evidence):
    return _NigHead.apply(evidence)


_edges_cache = {}


_const_cache = {}


def constant(value: float, shape, device) -> torch.Tensor:
    """A cached read-only constant tensor (attention weights that are identically 1, default masks / zero features): one
    fill when first requested instead of one at::fill kernel per forward.  Callers must not write to it."""
    key = (float(value), tuple(int(d) for d in shape), str(device))
    t = _const_cache.get(key)
    if t is None:
        t = _const_cache[key] = torch.full(key[1], float(value), device=device, dtype=torch.float32)
    return t


def ece_edges(device):
    """torch.linspace(0,1,11) exactly as losses.py:207 builds it (computed once on the host)."""
    key = str(device)
    if key not in _edges_cache:
        _edges_cache[key] = torch.linspace(0, 1, 11, dtype=torch.float32).to(device)
    return _edges_cache[key]


def _target_mask(target_mask, t: torch.Tensor) -> torch.Tensor:
    """Host-side checks of a target mask against targets `t` [B,D] (shape, dtype, device; the values are never read
    here, so a step with a mask stays graph-capturable)."""
    if not isinstance(target_mask, torch.Tensor) or not target_mask.is_cuda or target_mask.device != t.device:
        raise _lib.DeerError(f"deer_b200: `target_mask` must be a CUDA tensor on {t.device}")
    if target_mask.dtype not in (torch.bool, torch.uint8):
        raise _lib.DeerError(f"deer_b200: `target_mask` must be bool or uint8, got {target_mask.dtype}")
    if tuple(target_mask.shape) != tuple(t.shape):
        raise _lib.DeerError(f"deer_b200: `target_mask` must have the targets' shape {tuple(t.shape)}, got "
                             f"{tuple(target_mask.shape)}")
    return target_mask.contiguous()


def nig_loss_raw(evidence, params, targets, *, weights=(0.1, 0.01, 0.05, 0.05), eps=1e-8, task_weights=None,
                 want_nig=False, want_grad=True, grad_scale=1.0, stats_hook=None, global_batch=None, target_mask=None,
                 counts=None):
    """Fused DEER multitask loss on either raw evidence [B,D,4] or params=(gamma,nu,alpha,beta) each [B,D].

    Returns (losses [5D+2], grad, nig_out [7,B,D] or None, stats [D,40]).  `stats_hook(stats)` runs between the two
    phases (the data-parallel trainer all-reduces the statistics there).

    `target_mask` [B,D] (bool / uint8, CUDA; nonzero = labelled): partially labelled batch.  Each dimension's terms
    are means over its N_d labelled entries (N_d from the statistics, so after `stats_hook` it is the global count and
    `global_batch` is not used), the cross-dimension term covers the dimensions with N_d > 0, a dimension without labels
    has five 0 loss entries, and the gradient is exactly 0 at unlabelled entries, whatever their target values.
    `counts` (float32 [D], mask only) receives N_d."""
    from_ev = evidence is not None
    t = _req(targets, "targets").contiguous()
    B, D = t.shape
    dev = t.device
    m = None if target_mask is None else _target_mask(target_mask, t)
    if counts is not None and (m is None or _req(counts, "counts").shape != (D,)):
        raise _lib.DeerError(f"deer_b200: `counts` is a float32 [{D}] output of the target-mask path")
    if from_ev:
        e = _req(evidence, "evidence").contiguous()
        g = n = a = b = None
    else:
        e = None
        g, n, a, b = [_req(p, "nig param").contiguous() for p in params]
    stats = zeros_scratch((D, 40), dev)
    nig_out = torch.empty((7, B, D), device=dev, dtype=torch.float32) if want_nig else None
    edges = ece_edges(dev)
    if m is None:
        call("deer_nig_loss_stats", ptr(e), ptr(g), ptr(n), ptr(a), ptr(b), ptr(t), ptr(edges), ptr(stats),
             ptr(nig_out), B, D, int(from_ev), float(eps))
    else:
        call("deer_nig_loss_stats_mask", ptr(e), ptr(g), ptr(n), ptr(a), ptr(b), ptr(t), m.data_ptr(), ptr(edges),
             ptr(stats), ptr(nig_out), B, D, int(from_ev), float(eps))
    if stats_hook is not None:
        stats_hook(stats)
    losses = torch.empty(5 * D + 2, device=dev, dtype=torch.float32)
    grad = torch.empty((B, D, 4), device=dev, dtype=torch.float32) if want_grad else None
    tw = None if task_weights is None else torch.as_tensor(task_weights, dtype=torch.float32, device=dev)
    rw, kw, ew, cw = weights
    if m is None:
        call("deer_nig_loss_finish", ptr(e), ptr(g), ptr(n), ptr(a), ptr(b), ptr(t), ptr(edges), ptr(stats), ptr(tw),
             float(rw), float(kw), float(ew), float(cw), float(eps), B, int(global_batch or B), D, int(from_ev),
             float(grad_scale), ptr(losses), ptr(grad))
    else:
        call("deer_nig_loss_finish_mask", ptr(e), ptr(g), ptr(n), ptr(a), ptr(b), ptr(t), m.data_ptr(), ptr(edges),
             ptr(stats), ptr(tw), float(rw), float(kw), float(ew), float(cw), float(eps), B, D, int(from_ev),
             float(grad_scale), ptr(losses), ptr(grad), ptr(counts))
    return losses, grad, nig_out, stats


def _mask_counts(target_mask, targets):
    """The [D] output for N_d when a target mask is given (None otherwise)."""
    if target_mask is None:
        return None
    return torch.empty(targets.shape[-1], device=targets.device, dtype=torch.float32)


class _MultiTaskLoss(torch.autograd.Function):
    """losses.MultiTaskDEERLoss on contiguous [B,D] NIG parameter arrays.  Only `total` carries gradient."""

    @staticmethod
    def forward(ctx, gamma, nu, alpha, beta, targets, weights, eps, task_weights, target_mask=None):
        counts = _mask_counts(target_mask, targets)
        losses, grad, _, _ = nig_loss_raw(None, (gamma, nu, alpha, beta), targets, weights=weights, eps=eps,
                                          task_weights=task_weights, target_mask=target_mask, counts=counts)
        ctx.save_for_backward(grad)
        if counts is None:
            return losses
        ctx.mark_non_differentiable(counts)
        return losses, counts

    @staticmethod
    def backward(ctx, dlosses, *_dcounts):
        (grad,) = ctx.saved_tensors  # [B,D,4] = d total / d(gamma,nu,alpha,beta)
        D = grad.shape[1]
        s = dlosses[5 * D + 1]
        g = grad * s
        return g[..., 0], g[..., 1], g[..., 2], g[..., 3], None, None, None, None, None


def multitask_loss(gamma, nu, alpha, beta, targets, weights=(0.1, 0.01, 0.05, 0.05), eps=1e-8, task_weights=None,
                   target_mask=None):
    """losses [5D+2]; with `target_mask` [B,D] (see nig_loss_raw) the pair (losses, N_d [D])."""
    return _MultiTaskLoss.apply(gamma, nu, alpha, beta, targets, weights, eps, task_weights, target_mask)


class _FusedHeadLoss(torch.autograd.Function):
    """evidence [B,D,4] + targets -> (nig_out [7,B,D] (non-differentiable), losses [5D+2]); head and loss fused."""

    @staticmethod
    def forward(ctx, evidence, targets, weights, eps, task_weights, target_mask=None):
        counts = _mask_counts(target_mask, targets)
        losses, grad, nig_out, _ = nig_loss_raw(evidence, None, targets, weights=weights, eps=eps,
                                                task_weights=task_weights, want_nig=True, target_mask=target_mask,
                                                counts=counts)
        ctx.save_for_backward(grad)
        ctx.mark_non_differentiable(nig_out)
        if counts is None:
            return nig_out, losses
        ctx.mark_non_differentiable(counts)
        return nig_out, losses, counts

    @staticmethod
    def backward(ctx, _dnig, dlosses, *_dcounts):
        (grad,) = ctx.saved_tensors
        D = grad.shape[1]
        return grad * dlosses[5 * D + 1], None, None, None, None, None


def fused_head_loss(evidence, targets, weights=(0.1, 0.01, 0.05, 0.05), eps=1e-8, task_weights=None,
                    target_mask=None):
    """(nig_out, losses); with `target_mask` [B,D] (see nig_loss_raw) (nig_out, losses, N_d [D]).  nig_out covers
    every entry, labelled or not."""
    return _FusedHeadLoss.apply(evidence, targets, weights, eps, task_weights, target_mask)


class _AminiLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, mu, nu, alpha, beta, targets, ew, kw):
        args = [_req(t, "nig").contiguous() for t in (mu, nu, alpha, beta)]
        t = _req(targets, "targets").contiguous()
        n = t.numel()
        dev = t.device
        losses = torch.empty(5, device=dev, dtype=torch.float32)
        dparams = torch.empty((4, n), device=dev, dtype=torch.float32)
        scratch = torch.empty(8, device=dev, dtype=torch.float32)
        call("deer_amini_loss", *[ptr(a) for a in args], ptr(t), float(ew), float(kw), n, ptr(losses), ptr(dparams),
             ptr(scratch))
        ctx.save_for_backward(dparams)
        ctx.shape = mu.shape
        return losses

    @staticmethod
    def backward(ctx, dl):
        (dp,) = ctx.saved_tensors
        g = dp * dl[0]
        sh = ctx.shape
        return g[0].view(sh), g[1].view(sh), g[2].view(sh), g[3].view(sh), None, None, None


def amini_loss(mu, nu, alpha, beta, targets, evidence_weight=1.0, kl_weight=1.0):
    return _AminiLoss.apply(mu, nu, alpha, beta, targets, evidence_weight, kl_weight)


# ----------------------------------------------------------------------------------------------- small combiners
class _Mix(torch.autograd.Function):
    """out = w[:,None]*s + (1-u[:,None])*c with w,u column views (complete_project.py:282-293)."""

    @staticmethod
    def forward(ctx, w, u, s, c):
        s, c = _req(s, "s").contiguous(), _req(c, "c").contiguous()
        M, N = s.shape
        out = torch.empty_like(s)
        call("deer_mix_fwd", ptr(w), w.stride(0), ptr(u), u.stride(0), ptr(s), ptr(c), ptr(out), M, N)
        ctx.save_for_backward(w, u, s, c)
        return out

    @staticmethod
    def backward(ctx, dout):
        w, u, s, c = ctx.saved_tensors
        M, N = s.shape
        dw = torch.empty(M, device=s.device, dtype=torch.float32)
        du = torch.empty(M, device=s.device, dtype=torch.float32)
        ds, dc = torch.empty_like(s), torch.empty_like(c)
        call("deer_mix_bwd", ptr(dout.contiguous()), ptr(w), w.stride(0), ptr(u), u.stride(0), ptr(s), ptr(c), ptr(dw),
             1, ptr(du), 1, ptr(ds), ptr(dc), M, N)
        return dw.view(w.shape), du.view(u.shape), ds, dc


def mix(w, u, s, c):
    return _Mix.apply(w, u, s, c)


class _Gate(torch.autograd.Function):
    @staticmethod
    def forward(ctx, g, a, b):
        g, a, b = [_req(t, "gate").contiguous() for t in (g, a, b)]
        out = torch.empty_like(a)
        call("deer_gate_fwd", ptr(g), ptr(a), ptr(b), ptr(out), a.numel())
        ctx.save_for_backward(g, a, b)
        return out

    @staticmethod
    def backward(ctx, dout):
        g, a, b = ctx.saved_tensors
        dg, da, db = torch.empty_like(g), torch.empty_like(a), torch.empty_like(b)
        call("deer_gate_bwd", ptr(dout.contiguous()), ptr(g), ptr(a), ptr(b), ptr(dg), ptr(da), ptr(db), a.numel())
        return dg, da, db


def gate(g, a, b):
    return _Gate.apply(g, a, b)


class _SoftmaxRows(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        x = _req(x, "x").contiguous()
        M, N = x.shape
        y = torch.empty_like(x)
        call("deer_softmax_rows_fwd", ptr(x), ptr(y), M, N)
        ctx.save_for_backward(y)
        return y

    @staticmethod
    def backward(ctx, dy):
        (y,) = ctx.saved_tensors
        M, N = y.shape
        dx = torch.empty_like(y)
        call("deer_softmax_rows_bwd", ptr(dy.contiguous()), ptr(y), ptr(dx), M, N)
        return dx


def softmax_rows(x):
    return _SoftmaxRows.apply(x)


class _ColDiv(torch.autograd.Function):
    """y[m,n] = x[m,n] / t[n]  (UncertaintyCalibrationLayer temperature scaling, complete_project.py:449)."""

    @staticmethod
    def forward(ctx, x, t):
        x = _req(x, "x").contiguous()
        M, N = x.shape
        y = torch.empty_like(x)
        call("deer_coldiv_fwd", ptr(x), ptr(t), ptr(y), M, N)
        ctx.save_for_backward(x, t)
        ctx.params = (t,)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, t = ctx.saved_tensors
        M, N = x.shape
        dx = torch.empty_like(x)
        dt, direct = _acc(ctx.params[0]) if ctx.needs_input_grad[1] else (None, False)
        call("deer_coldiv_bwd", ptr(dy.contiguous()), ptr(x), ptr(t), ptr(dx), ptr(dt), M, N)
        return dx, None if direct else dt


def coldiv(x, t):
    return _ColDiv.apply(x, t)


class _Add(torch.autograd.Function):
    """a + b through deer_axpby (residual connections, complete_project.py:73)."""

    @staticmethod
    def forward(ctx, a, b):
        a, b = _req(a, "a").contiguous(), _req(b, "b").contiguous()
        y = torch.empty_like(a)
        call("deer_axpby", ptr(a), ptr(b), ptr(y), a.numel(), 1.0, 1.0)
        return y

    @staticmethod
    def backward(ctx, dy):
        return dy, dy


def add(a, b):
    return _Add.apply(a, b)
