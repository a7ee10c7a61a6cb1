"""Drop-in for the reference's acoustic model, timit/models/model_ctc.py (BatchRNN :13-36,
LayerCNN :38-68, CTC_Model :70-229).

Same constructor arguments, attributes, `state_dict()` keys/shapes (`conv.{n}.conv.*`,
`conv.{n}.batch_norm.*`, `rnns.{l}.batch_norm.*`, `rnns.{l}.rnn.weight_{ih,hh}_l0[_reverse]`, `fc.*`)
and the same forward contract (x [N,T,F] f32 -> log-probs [T',N,C] f32, differentiable), but every FLOP
runs in libctcb200's sm_100a kernels: the input projections, weight gradients and the output layer on the
tcgen05 GEMM, the time recurrence in the persistent recurrent kernels, BatchNorm / LogSoftmax / layout
changes in the streaming kernels. The torch modules below are parameter containers only (so checkpoints
interchange with the reference); their forward() is never called.

Behaviour kept on purpose (SURVEY.md appendix A): the LSTM and BatchNorm run over all padded frames,
layer 0 never has BatchNorm, BatchNorm statistics are over T*N rows, the fc BatchNorm follows
rnn_param['batch_norm'].
"""
import contextlib
import ctypes
import math
import os
from collections import OrderedDict

import torch
import torch.nn as nn

from . import _lib
from . import ops

__all__ = ["BatchRNN", "LayerCNN", "CTC_Model"]


def _round_up(x, m):
    return (x + m - 1) // m * m


class BatchRNN(nn.Module):
    """Optional BatchNorm1d over the feature axis, a bidirectional bias-free LSTM, then dropout."""

    def __init__(self, input_size, hidden_size, rnn_type=nn.LSTM, bidirectional=False, batch_norm=True, dropout=0.1):
        super(BatchRNN, self).__init__()
        self.input_size = input_size
        self.hidden_size = hidden_size
        self.bidirectional = bidirectional
        self.batch_norm = nn.BatchNorm1d(input_size) if batch_norm else None
        self.rnn = rnn_type(input_size=input_size, hidden_size=hidden_size, bidirectional=bidirectional, bias=False)
        self.dropout = nn.Dropout(p=dropout)

    def forward(self, x):
        raise RuntimeError("BatchRNN is executed by CTC_Model's fused CUDA path; call the model, not the layer")


class LayerCNN(nn.Module):
    """Conv2d (+BatchNorm2d) + activation (+MaxPool2d) + dropout block of the optional CNN front."""

    def __init__(self, in_channel, out_channel, kernel_size, stride, padding, pooling_size=None,
                 activation_function=nn.ReLU, batch_norm=True, dropout=0.1):
        super(LayerCNN, self).__init__()
        if len(kernel_size) == 2:
            self.conv = nn.Conv2d(in_channel, out_channel, kernel_size=kernel_size, stride=stride, padding=padding)
            self.batch_norm = nn.BatchNorm2d(out_channel) if batch_norm else None
        else:
            self.conv = nn.Conv1d(in_channel, out_channel, kernel_size=kernel_size, stride=stride, padding=padding)
            self.batch_norm = nn.BatchNorm1d(out_channel) if batch_norm else None
        self.activation = activation_function(inplace=True)
        if pooling_size is not None and len(kernel_size) == 2:
            self.pooling = nn.MaxPool2d(pooling_size)
        elif len(kernel_size) == 1:
            self.pooling = nn.MaxPool1d(pooling_size)
        else:
            self.pooling = None
        self.dropout = nn.Dropout(p=dropout)

    def forward(self, x):
        raise RuntimeError("LayerCNN is executed by CTC_Model's CUDA path; call the model, not the layer")


# ----------------------------------------------------------------------------------------------------
# the fused RNN stack + output layer as one autograd node
# ----------------------------------------------------------------------------------------------------
class _Workspace(object):
    """Per-call tensors kept between forward and backward."""
    pass


def _call(name, *args):
    return _lib.lib().call(name, *args)


class _Opnd(object):
    """A GEMM operand: bf16 `hi`, plus the bf16 remainder `lo` in the split-operand ("x3") precision mode (else None)."""
    __slots__ = ("hi", "lo")

    def __init__(self, hi, lo=None):
        self.hi, self.lo = hi, lo

    def rows(self, a, b):
        return _Opnd(self.hi[a:b], None if self.lo is None else self.lo[a:b])

    def cols(self, a, b):
        return _Opnd(self.hi[:, a:b], None if self.lo is None else self.lo[:, a:b])


def _gemm(a, b, out=None, **kw):
    """C = A * B^T on the tcgen05 GEMM; in x3 mode the three products A_lo B_hi + A_hi B_lo + A_hi B_hi accumulate in fp32
    (the accumulating launches add their tiles into C through the TMA unit)."""
    if a.lo is None:
        return ops.gemm_tn(a.hi, b.hi, out=out, **kw)
    acc = bool(kw.pop("accumulate", False))
    out = ops.gemm_tn(a.lo, b.hi, out=out, accumulate=acc, **kw)
    ops.gemm_tn(a.hi, b.lo, out=out, accumulate=True, **kw)
    ops.gemm_tn(a.hi, b.hi, out=out, accumulate=True, **kw)
    return out


def _gemm_atb(a, b, out=None, **kw):
    """C = A^T * B, both operands with the contracted index as rows (the weight-gradient form, ops.gemm_atb); x3 mode: the same
    three accumulated products as _gemm."""
    if a.lo is None:
        return ops.gemm_atb(a.hi, b.hi, out=out, **kw)
    acc = bool(kw.pop("accumulate", False))
    out = ops.gemm_atb(a.lo, b.hi, out=out, accumulate=acc, **kw)
    ops.gemm_atb(a.hi, b.lo, out=out, accumulate=True, **kw)
    ops.gemm_atb(a.hi, b.hi, out=out, accumulate=True, **kw)
    return out


_GATE_PERM = {}


def _gate_row_perm(H, dev):
    """Row gather that turns a [4H, ...] matrix whose rows follow the recurrent kernels' packed gate order (unit block j, unit u,
    gate g -> row j*128 + u*4 + g: the column order of dG) into torch's order (row g*H + unit)."""
    key = (H, str(dev))
    if key not in _GATE_PERM:
        unit = torch.arange(H, device=dev)
        g = torch.arange(4, device=dev).view(4, 1)
        _GATE_PERM[key] = ((unit // 32) * 128 + (unit % 32) * 4 + g).reshape(-1)     # [4H]: index of torch row g*H + unit
    return _GATE_PERM[key]


# ----------------------------------------------------------------------------------------------------
# hidden sizes that are not a multiple of 128: every layer runs at Hp = 128 * ceil(H / 128) device units, the Hp - H extra units
# carry zero weights and stay exactly zero (DESIGN.md §3.2). Torch shapes (parameters, gradients, state_dict) keep H; activation
# and gradient buffers use the device layout, where the D*H real features of a layer output sit at columns d*Hp + unit.
# ----------------------------------------------------------------------------------------------------
MAX_HIDDEN = 1024        # largest device hidden size of the recurrent kernels
MAX_HIDDEN_X3 = 640      # ... in the split-operand mode (its W_lo slice and hi/lo operand image must fit shared memory)


def device_hidden(H):
    """Device hidden size the recurrent kernels run a layer of torch hidden size H at."""
    return _round_up(H, 128)


def check_hidden(H, x3):
    """Hidden sizes the recurrent kernels can run: a RuntimeError before anything is launched otherwise."""
    if H < 1:
        raise RuntimeError("rnn_hidden_size must be >= 1 (got %d)" % H)
    Hp = device_hidden(H)
    if Hp > MAX_HIDDEN:
        raise RuntimeError("rnn_hidden_size %d is not supported: the recurrent kernels run hidden sizes up to %d"
                           % (H, MAX_HIDDEN))
    if x3 and Hp > MAX_HIDDEN_X3:
        raise RuntimeError("precision='x3' runs hidden sizes up to %d (rnn_hidden_size %d runs at %d device units); use "
                           "precision='bf16' for larger layers" % (MAX_HIDDEN_X3, H, Hp))
    return Hp


_UNIT_COLS = {}


def unit_cols(H, Hp, D, dev):
    """Device column of every torch feature of a [*, D*H] layer output in the padded [*, D*Hp] layout: d*Hp + unit."""
    key = (H, Hp, D, str(dev))
    if key not in _UNIT_COLS:
        _UNIT_COLS[key] = (torch.arange(D, device=dev).view(D, 1) * Hp + torch.arange(H, device=dev)).reshape(-1)
    return _UNIT_COLS[key]


def pad_cols(w, cols, width):
    """fp32 copy of w [..., D*H] with its columns scattered to `cols` of a zero [..., width] tensor."""
    out = torch.zeros(w.shape[:-1] + (width,), dtype=torch.float32, device=w.device)
    out.index_copy_(w.dim() - 1, cols, w.detach().float())
    return out


def _cast_t(src, s_outer, s_inner, n_inner, R, C, scale=None, shift=None, want=True, want_t=False, x3=False):
    """fp32 (strided rows) -> bf16 [R, Cp] and/or bf16 [C, (R/n_inner)*n_pad] with the batch axis padded to 8; returns
    (_Opnd or None, _Opnd or None). x3: every output also gets its remainder part."""
    dev = src.device
    Cp = _round_up(C, 8)
    n_pad = _round_up(n_inner, 8) if n_inner > 1 else 1
    Rp = _round_up((R // n_inner) * n_pad, 8)
    outs = []
    for part in ((0, 1) if x3 else (0,)):
        dst = None
        if want:
            dst = (torch.empty if Cp == C else torch.zeros)((R, Cp), dtype=torch.bfloat16, device=dev)
        dst_t = None
        if want_t:
            alloc = torch.empty if (n_pad == n_inner and Rp == R) else torch.zeros
            dst_t = alloc((C, Rp), dtype=torch.bfloat16, device=dev)
        _call("ctcb200_cast_transpose", _lib.ptr(src), s_outer, s_inner, n_inner, _lib.ptr(scale), _lib.ptr(shift),
              _lib.ptr(dst), Cp, _lib.ptr(dst_t), Rp, n_pad, R, C, part, _lib.stream())
        outs.append((dst, dst_t))
    X = _Opnd(outs[0][0], outs[1][0] if x3 else None) if want else None
    XT = _Opnd(outs[0][1], outs[1][1] if x3 else None) if want_t else None
    return X, XT


_SIDE_STREAMS = {}


def _side_stream(dev):
    """Per-device side stream for work that is off the backward pass's critical path (weight-gradient GEMMs)."""
    key = dev.index if dev.index is not None else torch.cuda.current_device()
    if key not in _SIDE_STREAMS:
        _SIDE_STREAMS[key] = torch.cuda.Stream(device=dev)
    return _SIDE_STREAMS[key]


_RESIDENT = {}


def _resident_state(dev):
    """[uint32[2] device counter, host-side expected value] for the BPTT 'grid is resident' notifications."""
    key = dev.index if dev.index is not None else torch.cuda.current_device()
    if key not in _RESIDENT:
        _RESIDENT[key] = [torch.zeros(2, dtype=torch.int32, device=dev), 0]
    return _RESIDENT[key]


_RESIDENT_EVENTS = {}


def _resident_event(dev):
    """Per-device cudaEvent (timing disabled) the BPTT launch fires, as a programmatic event, once all of its blocks have
    started. Returns (torch event, raw handle)."""
    key = dev.index if dev.index is not None else torch.cuda.current_device()
    if key not in _RESIDENT_EVENTS:
        ev = torch.cuda.Event(enable_timing=False)
        ev.record(torch.cuda.current_stream(dev))   # materialises the underlying cudaEvent_t
        _RESIDENT_EVENTS[key] = ev
    ev = _RESIDENT_EVENTS[key]
    return ev, ctypes.c_void_p(ev.cuda_event)


def _overlap_gate():
    """How the side stream learns that the BPTT grid is resident.
    'memop': counter bumped by the kernel + cuStreamWaitValue32 — precise: the weight-gradient work of layer l starts the moment
             the BPTT grid of layer l-1 is resident (profiles/timeline_r2_cfg2_g2_memopgate.json).
    'event': programmatic launch event + cudaStreamWaitEvent — an ordinary stream dependency, but CUDA only guarantees that it is
             observed *no earlier* than the trigger: measured on B200 (profiles/timeline_r2_cfg2_g2_eventgate.json) it is observed
             when the BPTT kernel ENDS, so every layer's weight gradients run one layer late and two layers' worth is left for
             the tail of the backward pass (2-GPU cfg2 step 14.9 ms vs 13.75 ms with the memop gate).
    Default: memop everywhere. Round 1 saw one stall of a 2-GPU run with the memop gate and fell back to the event gate for
    world_size > 1; it never reproduced (round 2: 3 x 33 steps + a profiled run at 2 GPUs, SCALE runs at 4 / 8 GPUs), and the
    wait is on a counter that the kernel launched just before it on the main stream always bumps. CTCB200_OVERLAP_GATE
    overrides."""
    g = os.environ.get("CTCB200_OVERLAP_GATE")
    if g in ("event", "memop"):
        return g
    return "memop"


def _overlap_enabled(model):
    """Weight-gradient work on a side stream under the BPTT kernels (CTC_Model.overlap_wgrad, env override).

    See _overlap_gate() for the two gating mechanisms. CTCB200_OVERLAP_WGRAD=0/1 overrides."""
    env = os.environ.get("CTCB200_OVERLAP_WGRAD")
    if env is not None:
        return env == "1"
    return bool(getattr(model, "overlap_wgrad", True))


_GX_READY = {}


def _gx_ready_state(dev):
    """[uint32[1] device word, host-side base value] the side stream publishes the input projection's chunk count through."""
    key = dev.index if dev.index is not None else torch.cuda.current_device()
    if key not in _GX_READY:
        _GX_READY[key] = [torch.zeros(1, dtype=torch.int32, device=dev), 0]
    return _GX_READY[key]


_CONCURRENT = {}


def _streams_overlap(dev):
    """True when a kernel on the side stream runs while a kernel on the main stream is resident on `dev` (once per device and
    process). The streamed input projection launches a kernel that waits for later launches of another stream: under a tool that
    serialises kernels (Nsight Compute, CUDA_LAUNCH_BLOCKING, anything injected through CUDA_INJECTION64_PATH) it would wait for
    its timeout trap, so those cases keep the whole-projection form. ctcb200_concurrency_probe (include/ctcb200.h) measures what
    the environment variables cannot tell."""
    key = dev.index if dev.index is not None else torch.cuda.current_device()
    if key not in _CONCURRENT:
        ok = True
        for var in ("CUDA_INJECTION64_PATH", "NV_COMPUTE_PROFILER_PERFWORKS_DIR", "NV_NSIGHT_INJECTION_PORT_BASE"):
            if os.environ.get(var):
                ok = False
        if os.environ.get("CUDA_LAUNCH_BLOCKING", "0") not in ("", "0"):
            ok = False
        if ok:
            main_s, side_s = torch.cuda.current_stream(dev), _side_stream(dev)
            ok = _lib.lib().dll.ctcb200_concurrency_probe(ctypes.c_void_p(main_s.cuda_stream), ctypes.c_void_p(side_s.cuda_stream), 20) == 1
        _CONCURRENT[key] = ok
    return _CONCURRENT[key]


def _gx_stream_plan(model, T, N, H, x3, cell, packed, dev):
    """Streamed input projection (include/ctcb200.h, ctcb200_lstm_fwd_streamed): only the first time chunk of Gx = X W_ih^T is
    computed before the recurrent kernel starts; the other chunks are GEMM launches on the side stream, on the SMs the
    latency-bound recurrence leaves idle, published chunk by chunk through a stream memory operation the kernel polls.
    Returns None (whole projection first) or (chunks, chunk_T, side_ctas, mode) with mode 'stream' or 'serial' (same chunk
    launches, all before the recurrent kernel: the CPU emulation and CTCB200_OVERLAP_GX=serial).
    model.overlap_gx / CTCB200_OVERLAP_GX=0|1|serial, model.gx_chunks / CTCB200_GX_CHUNKS (default 8)."""
    env = os.environ.get("CTCB200_OVERLAP_GX")
    on = bool(getattr(model, "overlap_gx", True)) if env is None else env != "0"
    if not on or packed or T < 4:
        return None
    chunks = int(os.environ.get("CTCB200_GX_CHUNKS", getattr(model, "gx_chunks", 8)))
    chunk_T = max(2, -(-T // max(1, chunks)))   # (the kernels prefetch two steps ahead: chunk 0 must hold steps 0 and 1)
    chunks = -(-T // chunk_T)
    if chunks < 2:
        return None
    if dev.type != "cuda" or env == "serial":
        return chunks, chunk_T, 0, "serial"
    if _lib._DEBUG_SYNC or _overlap_gate() != "memop":
        return None   # a host synchronize between the launch and its chunks would never return
    ctas = int(_lib.lib().dll.ctcb200_lstm_fwd_ctas(N, H, int(model.batch_tile), 1 if x3 else 0, int(cell)))
    free = torch.cuda.get_device_properties(dev).multi_processor_count - ctas
    if ctas <= 0 or free < 16:
        return None   # not one all-resident clustered launch, or no SMs left for the GEMMs
    if not _streams_overlap(dev):
        return None   # kernels of two streams do not overlap here (profiler, blocking launches): the kernel would wait forever
    # The recurrent kernel will WAIT for the chunk GEMMs: none of them may be a kernel's first launch on this device (CUDA's
    # lazy loading of a kernel can wait for the running recurrent kernel — a deadlock in the first step of a fresh process).
    # ctcb200_lstm_fwd_streamed does this as well; doing it here keeps the load out of the launch sequence.
    _call("ctcb200_gemm_preload")
    return chunks, chunk_T, free, "stream"


_DG_PROGRESS = {}


def _dg_progress_state(dev):
    """[uint32[1] device counter, host-side base] the BPTT kernels count their finished gate-gradient chunks in."""
    key = dev.index if dev.index is not None else torch.cuda.current_device()
    if key not in _DG_PROGRESS:
        _DG_PROGRESS[key] = [torch.zeros(1, dtype=torch.int32, device=dev), 0]
    return _DG_PROGRESS[key]


def _dg_stream_plan(model, T, N, H, D, x3, cell, packed, overlap, dev):
    """Streamed gate gradients (include/ctcb200.h, ctcb200_lstm_bwd_streamed): the input-gradient GEMM dX = dG W_ih of a layer —
    and the weight-gradient contractions of the FIRST layer, which have no later BPTT kernel to hide under — follow the BPTT
    kernel chunk by chunk on the side stream instead of starting when it ends; only the last chunk is left for the main
    stream. Returns None or (chunks, chunk_T, ctas, mode), mode 'stream' or 'serial' (same chunk launches after the kernel: the
    CPU emulation and CTCB200_OVERLAP_DG=serial). model.overlap_dg / CTCB200_OVERLAP_DG=0|1|serial|force, model.dg_chunks /
    CTCB200_DG_CHUNKS (default 8). On the GPU the split-operand mode keeps the whole-GEMM path unless forced: its three products
    per contraction already fill the idle SMs for longer than a BPTT kernel runs."""
    env = os.environ.get("CTCB200_OVERLAP_DG")
    on = bool(getattr(model, "overlap_dg", True)) if env is None else env != "0"
    if not on or packed or D != 2 or T < 4:
        return None
    chunks = int(os.environ.get("CTCB200_DG_CHUNKS", getattr(model, "dg_chunks", 8)))
    chunk_T = max(1, -(-T // max(1, chunks)))
    chunks = -(-T // chunk_T)
    if chunks < 2:
        return None
    if dev.type != "cuda" or env == "serial":
        return chunks, chunk_T, 0, "serial"
    if (x3 and env != "force") or not overlap or _lib._DEBUG_SYNC or _overlap_gate() != "memop":
        return None
    ctas = int(_lib.lib().dll.ctcb200_lstm_bwd_plan(N, H, int(model.batch_tile), 1 if x3 else 0, int(cell)))
    if ctas <= 0:
        return None
    return chunks, chunk_T, ctas, "stream"


def _dropout_mask(model, shape, p, dev):
    """uint8 keep-mask for nn.Dropout(p). `model.mask_source(shape, p, device)` (tests: masks shared with the oracle)
    replaces the framework RNG when set."""
    src = getattr(model, "mask_source", None)
    if src is not None:
        return src(shape, p, dev).to(device=dev, dtype=torch.uint8).contiguous()
    return (torch.rand(shape, device=dev) >= p).to(torch.uint8)


def _inv_keep(p):
    return 0.0 if p >= 1.0 else 1.0 / (1.0 - p)


def _unwrap(mod):
    """my_863_corpus wraps BatchNorm / the output layer in SequenceWise (`.module`); timit/ uses the modules directly."""
    return mod.module if (mod is not None and hasattr(mod, "module") and not isinstance(mod, (nn.BatchNorm1d, nn.Linear, nn.Sequential))) else mod


def _cell_of(rnn):
    """(cell code of the C ABI, gate rows per unit in torch's weights) for a recurrent module the reference may build
    (train_ctc.py:20 supported_rnn): nn.LSTM -> (0, 4), nn.GRU -> (1, 3), nn.RNN tanh / relu -> (2 / 3, 1)."""
    if isinstance(rnn, nn.LSTM):
        return 0, 4
    if isinstance(rnn, nn.GRU):
        return 1, 3
    if isinstance(rnn, nn.RNN):
        return (3 if rnn.nonlinearity == "relu" else 2), 1
    raise RuntimeError("the B200 path implements nn.LSTM / nn.GRU / nn.RNN layers (got %r)" % (type(rnn),))


def _layer_dropout_p(layer):
    d = getattr(layer, "dropout", None)
    return float(d.p) if isinstance(d, nn.Dropout) else 0.0


def _realign(src, lengths, T, N, W, split, direction, dst=None, accumulate=False):
    """Move [T, N, W] rows between the left- and right-aligned layouts of a packed batch / zero its padding rows."""
    if dst is None:
        dst = torch.empty_like(src)
    _call("ctcb200_realign_rows", _lib.ptr(src), _lib.ptr(dst), _lib.ptr(lengths), T, N, W, split, direction,
          1 if accumulate else 0, _lib.stream())
    return dst


class _BNState(object):
    __slots__ = ("mean", "rstd", "scale", "shift", "batch", "gamma", "cols")


def _bn_prepare(bn, x2d, R, C, training, n_valid=0, cols=None):
    """Statistics (training) or running-stat affine (eval) for BatchNorm1d `bn` over rows of x2d [R, C]. n_valid > 0: packed
    mode, the statistics are over that many valid rows (the padding rows of x2d are zero). cols: device column of every torch
    feature (padded hidden size, see unit_cols): the kernels then see a [C] parameter image with gamma = beta = 0 on the padding
    columns, so scale = shift = 0 there, and only the torch buffers' own columns of the running statistics are updated."""
    dev = x2d.device
    st = _BNState()
    st.scale = torch.empty(C, dtype=torch.float32, device=dev)
    st.shift = torch.empty(C, dtype=torch.float32, device=dev)
    st.cols = cols
    gamma = bn.weight if bn.affine else None
    beta = bn.bias if bn.affine else None
    run_mean, run_var = bn.running_mean, bn.running_var
    if cols is not None:
        Cr = cols.numel()
        gamma = pad_cols(gamma if gamma is not None else torch.ones(Cr, device=dev), cols, C)
        beta = pad_cols(beta if beta is not None else torch.zeros(Cr, device=dev), cols, C)
        if run_mean is not None:
            run_mean, run_var = pad_cols(run_mean, cols, C), pad_cols(run_var, cols, C)
    st.gamma = gamma if cols is not None else bn.weight
    use_batch = training or not bn.track_running_stats
    st.batch = use_batch
    if use_batch:
        st.mean = torch.empty(C, dtype=torch.float32, device=dev)
        st.rstd = torch.empty(C, dtype=torch.float32, device=dev)
        ws = torch.empty(2 * C, dtype=torch.float64, device=dev)
        upd = training and bn.track_running_stats
        mom = 0.1 if bn.momentum is None else float(bn.momentum)
        if upd:
            bn.num_batches_tracked.add_(1)
            if bn.momentum is None:
                mom = 1.0 / float(bn.num_batches_tracked.item())
        _call("ctcb200_bn_train_stats", _lib.ptr(x2d), R, C, _lib.ptr(gamma), _lib.ptr(beta),
              _lib.ptr(run_mean if upd else None), _lib.ptr(run_var if upd else None), mom,
              float(bn.eps), _lib.ptr(st.mean), _lib.ptr(st.rstd), _lib.ptr(st.scale), _lib.ptr(st.shift),
              _lib.ptr(ws), int(n_valid), _lib.stream())
        if upd and cols is not None:
            bn.running_mean.copy_(run_mean.index_select(0, cols))
            bn.running_var.copy_(run_var.index_select(0, cols))
    else:
        # frozen statistics (eval mode): the same per-column affine; mean / rstd kept for a possible backward pass
        st.mean = run_mean.detach().float().contiguous()
        st.rstd = torch.rsqrt(run_var.detach().float() + float(bn.eps)).contiguous()
        _call("ctcb200_bn_eval_affine", _lib.ptr(gamma), _lib.ptr(beta), _lib.ptr(run_mean),
              _lib.ptr(run_var), float(bn.eps), _lib.ptr(st.scale), _lib.ptr(st.shift), C, _lib.stream())
    return st


def _packed_weights(model, li, rnn, H, I, Ipad, x3, dev, Hp=None, Ir=None, i_blk=None):
    """bf16 operand layouts of one layer's four weight matrices (hi, and lo in x3 mode). Re-packed only when a parameter
    changed since the last call (inference / evaluation loops reuse them; an optimizer step bumps the version counters).
    Padded hidden size (Hp > H): the layouts are built at Hp from the torch-shaped weights (ctcb200_pack_lstm_weights_padded);
    I is then the device input width, Ir the torch one, and the input columns come in blocks of i_blk spread Hp apart above
    the first layer."""
    uni = not hasattr(rnn, "weight_ih_l0_reverse")
    if uni:
        # unidirectional layer (rnn_param["bidirectional"] = False): the kernels always run both directions of a layer
        # side by side on disjoint SMs, so the forward-only layer is the same launch with ZERO reverse weights — the reverse
        # half computes h = 0 and is dropped; no extra time on the recurrence's critical path
        zi = model.__dict__.setdefault("_zero_rev", {}).get((li, str(dev)))
        if zi is None:
            zi = (torch.zeros_like(rnn.weight_ih_l0), torch.zeros_like(rnn.weight_hh_l0))
            model.__dict__["_zero_rev"][(li, str(dev))] = zi
        wih_r, whh_r = zi
    else:
        wih_r, whh_r = rnn.weight_ih_l0_reverse, rnn.weight_hh_l0_reverse
    key = (x3, rnn.weight_ih_l0._version, rnn.weight_hh_l0._version, wih_r._version, whh_r._version,
           rnn.weight_ih_l0.data_ptr(), str(dev))
    cache = model.__dict__.setdefault("_pack_cache", {})
    ent = cache.get(li)
    if ent is not None and ent[0] == key:
        return ent[1]
    parts = []
    pad = Hp is not None and Hp != H
    Hd = Hp if pad else H
    for part in ((0, 1) if x3 else (0,)):
        wih_p = torch.empty((8 * Hd, Ipad), dtype=torch.bfloat16, device=dev)
        wihT_p = torch.empty((I, 8 * Hd), dtype=torch.bfloat16, device=dev)
        whh_p = torch.empty((8 * Hd, Hd), dtype=torch.bfloat16, device=dev)
        whhT_p = torch.empty((8 * Hd, Hd), dtype=torch.bfloat16, device=dev)
        if pad:
            blk = i_blk if i_blk is not None else Ir
            _call("ctcb200_pack_lstm_weights_padded", _lib.ptr(rnn.weight_ih_l0), _lib.ptr(rnn.weight_hh_l0),
                  _lib.ptr(wih_r), _lib.ptr(whh_r), _lib.ptr(wih_p), _lib.ptr(wihT_p), _lib.ptr(whh_p), _lib.ptr(whhT_p),
                  H, Hp, Ir, blk, Hp if i_blk is not None else blk, Ipad, part, _cell_of(rnn)[1], _lib.stream())
        else:
            _call("ctcb200_pack_lstm_weights", _lib.ptr(rnn.weight_ih_l0), _lib.ptr(rnn.weight_hh_l0),
                  _lib.ptr(wih_r), _lib.ptr(whh_r), _lib.ptr(wih_p),
                  _lib.ptr(wihT_p), _lib.ptr(whh_p), _lib.ptr(whhT_p), H, I, Ipad, part, _cell_of(rnn)[1], _lib.stream())
        parts.append((wih_p, wihT_p, whh_p, whhT_p))
    packed = tuple(_Opnd(parts[0][i], parts[1][i] if x3 else None) for i in range(4))
    cache[li] = (key, packed)
    return packed


class _RnnStackFn(torch.autograd.Function):
    """x [T*N rows as (t,n), I0] view of the input -> log-probs [T, N, C]."""

    @staticmethod
    def forward(ctx, model, x_src, geom, *params):
        # geom: (T, N, I0, s_outer, s_inner, need_grad[, lengths, raw_out]) describing where row (t, n) of the layer-0 input
        # lives in x_src; lengths (i64 [N] on the device, or None) switches on packed-sequence semantics (my_863_corpus),
        # raw_out returns the output layer's activations instead of log-probabilities (warp-ctc applies softmax itself)
        T, N, I0, s_outer, s_inner, need_grad = geom[:6]
        lengths = geom[6] if len(geom) > 6 else None
        raw_out = bool(geom[7]) if len(geom) > 7 else False
        packed = lengths is not None
        n_valid = int(geom[8]) if packed else 0
        dev = x_src.device
        training = model.training
        x3 = model.precision == "x3"
        R = T * N
        H = model.rnn_param["rnn_hidden_size"]   # torch shapes
        Hp = check_hidden(H, x3)                  # device layouts (Hp > H: zero-padded units, see device_hidden)
        pad = Hp != H
        C = model.num_class
        D = 2 if model.rnn_param["bidirectional"] else 1   # D = 1: forward half only (see _packed_weights)
        if packed and D == 1:
            raise RuntimeError("the packed-sequence path implements bidirectional layers only")
        cols = unit_cols(H, Hp, D, dev) if pad else None   # device column of each torch feature of a layer output
        layers = list(model.rnns.children())
        ws = _Workspace()
        ws.geom, ws.layers_n, ws.x3, ws.D = geom, len(layers), x3, D
        ws.lengths, ws.n_valid, ws.raw_out = lengths, n_valid, raw_out
        ws.L = []
        stream = _lib.stream

        scratch = torch.empty(_lib.lib().dll.ctcb200_lstm_scratch_bytes(N, Hp), dtype=torch.uint8, device=dev)
        # Weight gradients contract over the T*N rows: the tensor-core GEMM takes both operands in that (MN-major) form
        # (ops.gemm_atb), so the bf16 operands the forward pass makes anyway are kept and no transposed copies are built.
        defer_t = need_grad and _overlap_enabled(model) and not packed   # overlapped weight-gradient pipeline in backward()
        ws.defer_t = defer_t
        if packed:
            # layer-0 input as a dense time-major [T, N, I0] tensor with zero padding, plus its right-aligned twin
            if s_outer != N * I0 or s_inner != I0 or not x_src.is_contiguous():
                raise RuntimeError("packed mode takes the input as a contiguous time-major [T, N, F] tensor")
            x_l = _realign(x_src, lengths, T, N, I0, I0, 1)       # padding rows zeroed
            x_r = _realign(x_l, lengths, T, N, I0, 0, -1)
            X, _ = _cast_t(x_l, N * I0, I0, N, R, I0, want=True, want_t=False, x3=x3)
            Xr, _ = _cast_t(x_r, N * I0, I0, N, R, I0, want=True, want_t=False, x3=x3)
            del x_r
        else:
            X, _ = _cast_t(x_src, s_outer, s_inner, N, R, I0, want=True, want_t=False, x3=x3)
            Xr = None
        h_prev = None
        I = I0
        for li, layer in enumerate(layers):
            rec = _Workspace()
            rec.I = rec.Ir = I
            rec.bn = None
            layer_bn = _unwrap(layer.batch_norm)
            if li > 0:
                I = D * Hp
                rec.I, rec.Ir = I, D * H
                h_prev_r = _realign(h_prev, lengths, T, N, I, 0, -1) if packed else None
                if layer_bn is not None:
                    rec.bn = _bn_prepare(layer_bn, h_prev, R, I, training, n_valid, cols)
                    sc_, sh_ = rec.bn.scale, rec.bn.shift
                else:
                    sc_ = sh_ = None
                X, _ = _cast_t(h_prev, N * I, I, N, R, I, sc_, sh_, True, False, x3)
                if packed:   # the BatchNorm affine turns zero padding into `shift`: harmless, those rows are never consumed
                    Xr, _ = _cast_t(h_prev_r, N * I, I, N, R, I, sc_, sh_, True, False, x3)
                    del h_prev_r
            Ipad = _round_up(I, 8)
            wih_p, wihT_p, whh_p, whhT_p = _packed_weights(model, li, layer.rnn, H, I, Ipad, x3, dev, Hp, rec.Ir,
                                                           H if li > 0 else None)
            cell, G = _cell_of(layer.rnn)
            rec.cell, rec.G = cell, G
            hout = torch.empty((R, 2 * Hp), dtype=torch.float32, device=dev)
            c_save = torch.empty((R, 2 * Hp), dtype=torch.float32, device=dev) if need_grad else None
            gates = torch.empty((R, 2 * Hp, 4), dtype=torch.float32 if x3 else torch.float16, device=dev) if need_grad else None
            plan = _gx_stream_plan(model, T, N, Hp, x3, cell, packed, dev)
            if plan is None:
                if packed:   # each direction's input projection on its own alignment, written into its half of gx
                    gx = torch.empty((R, 8 * Hp), dtype=torch.float32, device=dev)
                    _gemm(X, wih_p.rows(0, 4 * Hp), out=gx[:, :4 * Hp], k=I)
                    _gemm(Xr, wih_p.rows(4 * Hp, 8 * Hp), out=gx[:, 4 * Hp:], k=I)
                else:
                    gx = _gemm(X, wih_p, k=I)  # [R, 8H] f32
                _call("ctcb200_lstm_fwd", _lib.ptr(gx), _lib.ptr(whh_p.hi), _lib.ptr(whh_p.lo), _lib.ptr(hout), _lib.ptr(c_save),
                      _lib.ptr(gates), _lib.ptr(scratch), T, N, Hp, model.batch_tile, cell, stream())
            else:
                # streamed input projection: chunk c = the rows each direction visits in its scan steps [c*chunk_T, ...)
                chunks, chunk_T, side_ctas, mode = plan
                gx = torch.empty((R, 8 * Hp), dtype=torch.float32, device=dev)

                def _gx_chunk(c, mc):
                    a, b = c * chunk_T, min(T, (c + 1) * chunk_T)
                    for d, (r0, r1) in enumerate(((a * N, b * N), ((T - b) * N, (T - a) * N))):
                        _gemm(X.rows(r0, r1), wih_p.rows(d * 4 * Hp, (d + 1) * 4 * Hp),
                              out=gx[r0:r1, d * 4 * Hp:(d + 1) * 4 * Hp], k=I, max_ctas=mc)

                _gx_chunk(0, 0)
                if mode == "serial":
                    for c in range(1, chunks):
                        _gx_chunk(c, 0)
                    _call("ctcb200_lstm_fwd", _lib.ptr(gx), _lib.ptr(whh_p.hi), _lib.ptr(whh_p.lo), _lib.ptr(hout),
                          _lib.ptr(c_save), _lib.ptr(gates), _lib.ptr(scratch), T, N, Hp, model.batch_tile, cell, stream())
                else:
                    main_s, side_s = torch.cuda.current_stream(dev), _side_stream(dev)
                    res, rdy = _resident_state(dev), _gx_ready_state(dev)
                    base = rdy[1]
                    rdy[1] = (base + chunks) & 0xFFFFFFFF
                    x_ready = torch.cuda.Event()
                    x_ready.record(main_s)
                    _call("ctcb200_lstm_fwd_streamed", _lib.ptr(gx), _lib.ptr(whh_p.hi), _lib.ptr(whh_p.lo), _lib.ptr(hout),
                          _lib.ptr(c_save), _lib.ptr(gates), _lib.ptr(scratch), T, N, Hp, model.batch_tile, cell,
                          _lib.ptr(res[0]), _lib.ptr(rdy[0]), base, chunk_T, stream())
                    res[1] = (res[1] + 1) & 0xFFFFFFFF
                    with torch.cuda.stream(side_s):
                        side_s.wait_event(x_ready)
                        # the recurrent grid is resident: its clusters can no longer be blocked by GEMM CTAs
                        _call("ctcb200_stream_wait_geq", _lib.stream(), _lib.ptr(res[0]), res[1])
                        for c in range(1, chunks):
                            _gx_chunk(c, side_ctas)
                            _call("ctcb200_stream_write_value", _lib.stream(), _lib.ptr(rdy[0]), (base + c) & 0xFFFFFFFF)
                    main_s.wait_stream(side_s)   # (already implied by the kernel's own waits; keeps the allocator's view simple)
            del gx
            rec.Hb = None
            p_drop = _layer_dropout_p(layer)
            # dW_hh pairs dG_t with the *pre-dropout* h_{t-1}: its bf16 copy can only be left to the backward pass when hout
            # is not modified in place
            if need_grad and training and p_drop > 0.0 and not packed:
                rec.Hb, _ = _cast_t(hout, N * 2 * Hp, 2 * Hp, N, R, 2 * Hp, want=True, want_t=False, x3=x3)
            rec.h_out = hout if need_grad else None
            if packed:
                # kernel alignment (forward half left-, reverse half right-aligned, garbage in the padding) -> left-aligned
                # layer output with zero padding: what pad_packed_sequence would show (my_863_corpus/steps/model.py:93-141)
                hout = _realign(hout, lengths, T, N, 2 * Hp, Hp, 1)
            if D == 1:
                hout = hout[:, :Hp].contiguous()    # the layer's output is the forward half
            rec.mask = None
            if training and p_drop > 0.0:
                rec.mask = _dropout_mask(model, (R, D * H), p_drop, dev)   # drawn in torch's shape whatever the layout
                if pad:
                    rec.mask = pad_cols(rec.mask, cols, D * Hp).to(torch.uint8)
                _call("ctcb200_dropout_apply", _lib.ptr(hout), _lib.ptr(rec.mask), _inv_keep(p_drop), hout.numel(), stream())
            rec.h_in = h_prev
            rec.Xb = X if need_grad else None
            rec.Xrb = Xr if (need_grad and packed) else None
            rec.c_save, rec.gates, rec.wihT_p, rec.whhT_p = c_save, gates, wihT_p, whhT_p
            ws.L.append(rec)
            h_prev = hout

        # output layer: (BatchNorm1d) + Linear(no bias) + LogSoftmax
        F2 = D * Hp
        fc = _unwrap(model.fc)
        fc_bn, fc_lin = (fc[0], fc[1]) if isinstance(fc, nn.Sequential) else (None, fc)
        C = fc_lin.weight.shape[0]
        ws.fc_bn = _bn_prepare(fc_bn, h_prev, R, F2, training, n_valid, cols) if fc_bn is not None else None
        Xfc, _ = _cast_t(h_prev, N * F2, F2, N, R, F2, ws.fc_bn.scale if ws.fc_bn else None,
                            ws.fc_bn.shift if ws.fc_bn else None, True, False, x3)
        ws.Xfc = Xfc if need_grad else None
        Wfc = pad_cols(fc_lin.weight, cols, F2) if pad else fc_lin.weight   # zero columns for the padding units
        Wfc_b, WfcT_b = _cast_t(Wfc, F2, F2, 1, C, F2, want=True, want_t=need_grad, x3=x3)
        logits = _gemm(Xfc, Wfc_b, k=F2)  # [R, C]
        if packed:   # after pad_packed_sequence every padded frame is a zero vector
            if logits.stride(0) != C:
                logits = logits.contiguous()
            _realign(logits, lengths, T, N, C, C, 1, dst=logits)
        if raw_out:
            out = logits.view(T, N, C) if logits.stride(0) == C else logits.contiguous().view(T, N, C)
        else:
            out = torch.empty((T, N, C), dtype=torch.float32, device=dev)
            _call("ctcb200_log_softmax_fwd", _lib.ptr(logits), logits.stride(0), _lib.ptr(out), R, C, stream())
        ws.h_last, ws.WfcT_b, ws.out = h_prev, WfcT_b, out
        ws.T, ws.N, ws.H, ws.Hp, ws.C, ws.R, ws.cols = T, N, H, Hp, C, R, cols
        ctx.ws = ws if need_grad else None
        ctx.model = model
        ctx.param_list = params
        return out

    @staticmethod
    def backward(ctx, g_out):
        ws, model = ctx.ws, ctx.model
        if ws is None:
            raise RuntimeError("backward through a forward pass that ran without gradient bookkeeping")
        T, N, H, C, R = ws.T, ws.N, ws.H, ws.C, ws.R   # H: torch shapes
        Hp, cols = ws.Hp, ws.cols                      # Hp: device layouts (cols: see unit_cols; None when Hp = H)
        x3, D = ws.x3, ws.D
        lengths, n_valid = ws.lengths, ws.n_valid
        packed = lengths is not None
        dev = g_out.device
        stream = _lib.stream
        F2, F2r = D * Hp, D * H
        layers = list(model.rnns.children())
        grads = {}
        grad_x = None
        main = torch.cuda.current_stream(dev)
        overlap = bool(ws.defer_t)
        side = _side_stream(dev) if overlap else None
        keep = []
        gate = _overlap_gate()
        sync = getattr(model, "grad_sync", None)   # data parallel: per-layer gradient all-reduce launched from in here
        if overlap:
            res = _resident_state(dev)
            gate_ev, gate_ev_ptr = _resident_event(dev)
            side_ctas = max(8, torch.cuda.get_device_properties(dev).multi_processor_count
                            - int(_lib.lib().dll.ctcb200_lstm_bwd_ctas(N, Hp, model.batch_tile)))
            if os.environ.get("CTCB200_SIDE_CTAS"):   # measurements: fewer CTAs for the side-stream GEMMs
                side_ctas = max(8, min(side_ctas, int(os.environ["CTCB200_SIDE_CTAS"])))

        def _flat(sizes):
            """One flat fp32 buffer per layer (views per parameter): its all-reduce is a single collective."""
            buf = torch.empty(sum(sizes), dtype=torch.float32, device=dev)
            views, off = [], 0
            for n_ in sizes:
                views.append(buf[off:off + n_])
                off += n_
            return buf, views

        g = g_out.detach().to(torch.float32).contiguous()
        if ws.raw_out:
            dlogits = g.view(R, C)
        else:
            dlogits = torch.empty((R, C), dtype=torch.float32, device=dev)
            _call("ctcb200_log_softmax_bwd", _lib.ptr(g), _lib.ptr(ws.out), _lib.ptr(dlogits), R, C, stream())
        if packed:   # nothing flows into padded frames
            dlogits = _realign(dlogits, lengths, T, N, C, C, 1)
        dLb, _ = _cast_t(dlogits, N * C, C, N, R, C, want=True, want_t=False, x3=x3)
        fc = _unwrap(model.fc)
        fc_bn, fc_lin = (fc[0], fc[1]) if isinstance(fc, nn.Sequential) else (None, fc)
        fc_buf, fc_views = _flat([C * F2r] + ([F2r, F2r] if fc_bn is not None else []))
        if cols is None:
            grads[fc_lin.weight] = _gemm_atb(dLb.cols(0, C), ws.Xfc.cols(0, F2), out=fc_views[0].view(C, F2), k=R)   # [C, 2H]
        else:   # padded layout: the torch columns of the product
            grads[fc_lin.weight] = torch.index_select(_gemm_atb(dLb.cols(0, C), ws.Xfc.cols(0, F2), k=R), 1, cols,
                                                      out=fc_views[0].view(C, F2r))
        dh = _gemm(dLb, ws.WfcT_b, k=C)                                                # [R, 2H]
        dws = torch.empty(2 * F2, dtype=torch.float64, device=dev)
        fuse_env = os.environ.get("CTCB200_BN_FUSE", "1") != "0"

        def _bn_backward(bn_mod, st, dy, x_in, C_, below, dgam, dbet):
            """BatchNorm1d backward of `bn_mod` for gradient dy [R, C_] w.r.t. its output; x_in is its input (the output of the
            layer below). Returns (bn_x, bn_coef) when the input gradient is left to the BPTT kernel of that layer (no dropout
            mask in between), else applies it in place and returns None. Padded layout: the kernels see the padded parameter
            image of _bn_prepare, dgam / dbet receive the torch columns."""
            grads[bn_mod.weight], grads[bn_mod.bias] = dgam, dbet
            if st.cols is None:
                return _bn_backward_dev(st, dy, x_in, C_, below, dgam, dbet)
            dgam_p = torch.empty(C_, dtype=torch.float32, device=dev)
            dbet_p = torch.empty(C_, dtype=torch.float32, device=dev)
            fused = _bn_backward_dev(st, dy, x_in, C_, below, dgam_p, dbet_p)
            torch.index_select(dgam_p, 0, st.cols, out=dgam)
            torch.index_select(dbet_p, 0, st.cols, out=dbet)
            return fused

        def _bn_backward_dev(st, dy, x_in, C_, below, dgam, dbet):
            if ((fuse_env and ws.L[below].mask is None and D == 2) or not st.batch) and not (packed and st.batch):
                coef = torch.empty(3 * C_, dtype=torch.float32, device=dev)
                _call("ctcb200_bn_bwd_coef", _lib.ptr(dy), _lib.ptr(x_in), _lib.ptr(st.mean), _lib.ptr(st.rstd),
                      _lib.ptr(st.gamma), _lib.ptr(coef), _lib.ptr(dgam), _lib.ptr(dbet), R, C_, _lib.ptr(dws), n_valid,
                      stream())
                if not st.batch:
                    coef[C_:].zero_()   # frozen statistics: dx = gamma * rstd * dy, no batch-coupling terms
                    if D == 1:          # no fused consumer for a half-width gradient: apply the scale here
                        dy.mul_(coef[:C_])
                        return None
                    if ws.L[below].mask is not None:   # (cannot happen: masks only exist in training mode)
                        raise RuntimeError("dropout mask together with frozen BatchNorm statistics")
                return (x_in, coef)
            # packed mode: the padding rows of dx come out non-zero here; the realign in front of the BPTT kernel zeroes them
            _call("ctcb200_bn_bwd", _lib.ptr(dy), _lib.ptr(x_in), _lib.ptr(st.mean), _lib.ptr(st.rstd),
                  _lib.ptr(st.gamma), _lib.ptr(dy), _lib.ptr(dgam), _lib.ptr(dbet), R, C_, _lib.ptr(dws), n_valid, stream())
            return None

        bn_fuse = None
        if fc_bn is not None:
            bn_fuse = _bn_backward(fc_bn, ws.fc_bn, dh, ws.h_last, F2, len(layers) - 1, fc_views[1], fc_views[2])
        if sync is not None:
            sync.reduce(fc_buf)   # the output layer's gradients travel while the whole RNN stack is still back-propagating

        def _wgrad_finish(item, tmp_ih, t1, t2, extra=()):
            """Weight-gradient products (rows in dG's packed gate order) -> torch's layout inside the layer's flat bucket; hands
            the bucket to the gradient all-reduce. Padded layout: the rows of the real units (the gate-row gather works at any
            Hp), then the torch columns (the padded input layout above the first layer, the real units of W_hh)."""
            layer_, rec_, (dg_, dgrec_), li_, buf_, views_ = item
            rnn = layer_.rnn
            GH = rec_.G * H     # rows of torch's weight matrices per direction (4H LSTM, 3H GRU, H RNN)
            I_ = rec_.Ir
            perm = _gate_row_perm(H, dev)
            in_cols = cols if (cols is not None and li_ > 0) else None
            hh_cols = unit_cols(H, Hp, 1, dev) if cols is not None else None

            def gather(src, out, col_idx):
                if col_idx is None:
                    torch.index_select(src, 0, perm, out=out)
                else:
                    torch.index_select(torch.index_select(src, 0, perm), 1, col_idx, out=out)
            dwih = views_[0].view(8 * H, I_)
            gather(tmp_ih[0], dwih[:4 * H], in_cols)
            gather(tmp_ih[1], dwih[4 * H:], in_cols)
            grads[rnn.weight_ih_l0] = dwih[:GH]
            whf, whr = views_[1].view(4 * H, H), views_[2].view(4 * H, H)
            if t1 is not None:
                gather(t1, whf, hh_cols)
            else:
                whf.zero_()
            if t2 is not None:
                gather(t2, whr, hh_cols)
            else:
                whr.zero_()
            grads[rnn.weight_hh_l0] = whf[:GH]
            if D == 2:
                grads[rnn.weight_ih_l0_reverse], grads[rnn.weight_hh_l0_reverse] = dwih[4 * H:4 * H + GH], whr[:GH]
            if sync is not None:
                sync.reduce(buf_)    # one collective per layer, behind the BPTT kernels of the layers below
            if torch.cuda.current_stream(dev) != main:  # allocated on the main stream, written here on the side stream
                buf_.record_stream(torch.cuda.current_stream(dev))
            keep.append((dg_, dgrec_, tmp_ih, t1, t2) + tuple(extra))  # alive until the streams are joined

        def _wgrad(item, mc):
            """dW_ih, dW_hh (both directions) of one layer from its gate gradients; runs on the current stream."""
            layer_, rec_, (dg_, dgrec_), li_, buf_, views_ = item
            I_ = rec_.I
            # contraction over the T*N rows with both operands as they are (ops.gemm_atb): gate gradients [R, 8H] from the
            # BPTT kernel, layer input [R, I] bf16 from the forward pass, layer output [R, 2H] cast here
            Xb, Hb = rec_.Xb, rec_.Hb
            if Hb is None:
                Hb, _ = _cast_t(rec_.h_out, N * 2 * Hp, 2 * Hp, N, R, 2 * Hp, want=True, want_t=False, x3=x3)
            if packed:   # each direction against the input in its own alignment
                tmp_ih = (_gemm_atb(dg_.cols(0, 4 * Hp), Xb.cols(0, I_), k=R, max_ctas=mc),
                          _gemm_atb(dg_.cols(4 * Hp, 8 * Hp), rec_.Xrb.cols(0, I_), k=R, max_ctas=mc))
            else:
                tmp = _gemm_atb(dg_, Xb.cols(0, I_), k=R, max_ctas=mc)                   # [8H, I]
                tmp_ih = (tmp[:4 * Hp], tmp[4 * Hp:])
            dgr_ = dgrec_ if dgrec_ is not None else dg_     # what the recurrent weights see (GRU differs)
            t1 = t2 = None
            if T > 1:
                # pairs (dG_t, h_{t-1}) for the forward scan, (dG_t, h_{t+1}) for the reverse scan: one time step = N rows
                t1 = _gemm_atb(dgr_.cols(0, 4 * Hp), Hb.cols(0, Hp), a_roff=N, b_roff=0, k=R - N, max_ctas=mc)
                if D == 2:
                    t2 = _gemm_atb(dgr_.cols(4 * Hp, 8 * Hp), Hb.cols(Hp, 2 * Hp), a_roff=0, b_roff=N, k=R - N, max_ctas=mc)
            _wgrad_finish(item, tmp_ih, t1, t2, (Xb, Hb))

        # ---- streamed gate gradients (_dg_stream_plan): chunk c = scan steps [c*chunk_T, (c+1)*chunk_T) of both BPTT scans ----
        def _chunk_frames(c, chunk_T):
            a, b = c * chunk_T, min(T, (c + 1) * chunk_T)
            return (T - b, T - a), (a, b)     # frames the forward direction's / the reverse direction's BPTT covers in chunk c

        def _dx_chunk(dg_, rec_, dx_, c, chunk_T, mc):
            """this chunk's share of dX = dG W_ih: each direction's K half against the rows it has finished (accumulated)."""
            for d, (ta, tb) in enumerate(_chunk_frames(c, chunk_T)):
                _gemm(dg_.rows(ta * N, tb * N), rec_.wihT_p, out=dx_[ta * N:tb * N], k=4 * Hp, a_koff=d * 4 * Hp,
                      b_koff=d * 4 * Hp, accumulate=True, max_ctas=mc)

        def _wg_chunk(st, c, chunk_T, mc):
            """this chunk's share of the first layer's dW_ih / dW_hh contractions over time (accumulated)."""
            dg_, dgr_, Xb, Hb, I_, tmp_ih, t1, t2 = st
            (fa, fb), (ra, rb) = _chunk_frames(c, chunk_T)
            _gemm_atb(dg_.cols(0, 4 * Hp), Xb.cols(0, I_), out=tmp_ih[0], accumulate=True, a_roff=fa * N, b_roff=fa * N,
                      k=(fb - fa) * N, max_ctas=mc)
            _gemm_atb(dg_.cols(4 * Hp, 8 * Hp), Xb.cols(0, I_), out=tmp_ih[1], accumulate=True, a_roff=ra * N, b_roff=ra * N,
                      k=(rb - ra) * N, max_ctas=mc)
            f0 = max(fa, 1)           # (dG_t, h_{t-1}), t >= 1
            if fb > f0:
                _gemm_atb(dgr_.cols(0, 4 * Hp), Hb.cols(0, Hp), out=t1, accumulate=True, a_roff=f0 * N, b_roff=(f0 - 1) * N,
                          k=(fb - f0) * N, max_ctas=mc)
            r1 = min(rb, T - 1)       # (dG_t, h_{t+1}), t <= T - 2
            if r1 > ra:
                _gemm_atb(dgr_.cols(4 * Hp, 8 * Hp), Hb.cols(Hp, 2 * Hp), out=t2, accumulate=True, a_roff=ra * N,
                          b_roff=(ra + 1) * N, k=(r1 - ra) * N, max_ctas=mc)

        pending = None
        scratch = torch.empty(_lib.lib().dll.ctcb200_lstm_scratch_bytes(N, Hp), dtype=torch.uint8, device=dev)
        for li in range(len(layers) - 1, -1, -1):
            layer, rec = layers[li], ws.L[li]
            I = rec.I
            layer_bn = _unwrap(layer.batch_norm)
            has_bn = li > 0 and layer_bn is not None
            Ir = rec.Ir
            buf, views = _flat([8 * H * Ir, 4 * H * H, 4 * H * H] + ([Ir, Ir] if has_bn else []))   # torch shapes
            if rec.mask is not None:
                _call("ctcb200_dropout_apply", _lib.ptr(dh), _lib.ptr(rec.mask), _inv_keep(_layer_dropout_p(layer)),
                      dh.numel(), stream())
            if packed:   # left-aligned gradient -> the kernels' alignment (reverse half right-aligned), padding rows zeroed
                dh = _realign(dh, lengths, T, N, 2 * Hp, Hp, -1)
            if D == 1:   # forward half only: the kernel still takes a [R, 2H] gradient, the reverse half gets none
                dh2 = torch.zeros((R, 2 * Hp), dtype=torch.float32, device=dev)
                dh2[:, :Hp].copy_(dh)
                dh = dh2
            def _dg_buf():
                # unused gate slots of GRU / RNN layers are never written by the kernel: they must read as zero
                alloc = torch.empty if rec.G == 4 else torch.zeros
                return _Opnd(alloc((R, 8 * Hp), dtype=torch.bfloat16, device=dev),
                             alloc((R, 8 * Hp), dtype=torch.bfloat16, device=dev) if x3 else None)
            dg = _dg_buf()
            dg_rec = _dg_buf() if rec.cell == 1 else None   # GRU: the recurrent weights see a different n-gate gradient
            need_dx = li > 0 or bool(ctx.needs_input_grad[1])
            plan = _dg_stream_plan(model, T, N, Hp, D, x3, rec.cell, packed, overlap and gate == "memop", dev)
            streamed = plan is not None and plan[3] == "stream"
            dx_s = wg0 = None
            if plan is not None:
                # streamed gate gradients: the chunk GEMMs accumulate into zero-initialised outputs (written on the main stream
                # before the BPTT launch, so they are ordered before every chunk on either stream)
                chunks, chunk_T, prog_ctas, _mode = plan
                if need_dx:
                    dx_s = torch.zeros((R, I), dtype=torch.float32, device=dev)
                if li == 0:   # the first layer's weight gradients have no later BPTT kernel to hide under
                    tmp0 = torch.zeros((8 * Hp, I), dtype=torch.float32, device=dev)
                    wg0 = [dg, dg_rec if dg_rec is not None else dg, rec.Xb, rec.Hb, I, (tmp0[:4 * Hp], tmp0[4 * Hp:]),
                           torch.zeros((4 * Hp, Hp), dtype=torch.float32, device=dev),
                           torch.zeros((4 * Hp, Hp), dtype=torch.float32, device=dev)]
            bwd_args = (_lib.ptr(dh), _lib.ptr(rec.whhT_p.hi), _lib.ptr(rec.whhT_p.lo), _lib.ptr(rec.c_save),
                        _lib.ptr(rec.gates), _lib.ptr(dg.hi), _lib.ptr(dg.lo), _lib.ptr(dg_rec.hi) if dg_rec else None,
                        _lib.ptr(dg_rec.lo) if dg_rec else None, _lib.ptr(scratch), T, N, Hp, model.batch_tile, rec.cell,
                        _lib.ptr(bn_fuse[0]) if bn_fuse else None, _lib.ptr(bn_fuse[1]) if bn_fuse else None,
                        _lib.ptr(res[0]) if (overlap and gate == "memop") else None)
            if streamed:
                prog = _dg_progress_state(dev)
                prog_base = prog[1]
                prog[1] = (prog_base + prog_ctas * chunks) & 0xFFFFFFFF
                _call("ctcb200_lstm_bwd_streamed", *(bwd_args + (_lib.ptr(prog[0]), chunk_T, stream())))
            else:
                _call("ctcb200_lstm_bwd", *(bwd_args + (gate_ev_ptr if (overlap and gate == "event") else None, stream())))
            if bn_fuse:
                keep.append(bn_fuse)
                bn_fuse = None
            # Weight gradients are not needed by the rest of the backward pass. Overlapped mode: those of the layer
            # above (its dG is complete) go to the side stream, gated on *this* layer's BPTT grid being resident, and
            # are confined to the SMs that latency-bound kernel leaves idle. The gate is only ever enqueued after the
            # launch it waits for.
            item = (layer, rec, (dg, dg_rec), li, buf, views)
            if overlap:
                if gate == "memop":
                    res[1] = (res[1] + 1) & 0xFFFFFFFF
                if pending is not None:
                    with torch.cuda.stream(side):
                        if pending[6] is not None:
                            side.wait_event(pending[6])   # this layer's BatchNorm gradients (main stream) share its bucket
                        if gate == "event":
                            side.wait_event(gate_ev)   # fires when every block of the BPTT grid just launched has started
                        else:
                            _call("ctcb200_stream_wait_geq", _lib.stream(), _lib.ptr(res[0]), res[1])
                        _wgrad(pending[:6], side_ctas)
                pending = None if wg0 is not None else [layer, rec, (dg, dg_rec), li, buf, views, None]

            def _chunks_of(c_list, mc):
                for c in c_list:
                    if streamed and mc:   # this chunk's rows of every CTA of the BPTT launch are written
                        _call("ctcb200_stream_wait_geq", _lib.stream(), _lib.ptr(prog[0]),
                              (prog_base + prog_ctas * (c + 1)) & 0xFFFFFFFF)
                    if dx_s is not None:
                        _dx_chunk(dg, rec, dx_s, c, chunk_T, mc)
                    if wg0 is not None:
                        _wg_chunk(wg0, c, chunk_T, mc)

            if plan is not None:
                if wg0 is not None and wg0[3] is None:
                    with torch.cuda.stream(side) if streamed else contextlib.nullcontext():
                        wg0[3], _ = _cast_t(rec.h_out, N * 2 * Hp, 2 * Hp, N, R, 2 * Hp, want=True, want_t=False, x3=x3)
                if streamed:
                    with torch.cuda.stream(side):
                        _chunks_of(range(chunks - 1), side_ctas)
                    main.wait_stream(side)
                    _chunks_of([chunks - 1], 0)   # the last chunk: behind the BPTT kernel on the main stream, on all SMs
                else:
                    _chunks_of(range(chunks), 0)
                if wg0 is not None:
                    _wgrad_finish(item, wg0[5], wg0[6], wg0[7], (wg0[2], wg0[3]))

            def _input_grad():
                if dx_s is not None:
                    return dx_s
                if not packed:
                    return _gemm(dg, rec.wihT_p, k=8 * Hp)                  # [R, I] rows (t, n)
                dxf = _gemm(dg, rec.wihT_p, k=4 * Hp)                       # forward direction: already left-aligned
                dxr = _gemm(dg, rec.wihT_p, k=4 * Hp, a_koff=4 * Hp, b_koff=4 * Hp)
                return _realign(dxr, lengths, T, N, I, 0, 1, dst=dxf, accumulate=True)
            if li == 0 and ctx.needs_input_grad[1]:
                dx0 = _input_grad()
                T0, N0, I0 = ws.geom[0], ws.geom[1], ws.geom[2]
                # back to the layout of x_src: [N, T, I0] for the padded model, time-major for the packed one
                grad_x = dx0.view(T0, N0, I0) if packed else dx0.view(T0, N0, I0).transpose(0, 1)
            if li > 0:
                dh = _input_grad()
                if has_bn:
                    bn_fuse = _bn_backward(layer_bn, rec.bn, dh, rec.h_in, I, li - 1, views[3], views[4])
                    if overlap and sync is not None and pending is not None:
                        pending[6] = torch.cuda.Event()
                        pending[6].record(main)
            if not overlap and wg0 is None:
                _wgrad(item, 0)
        if overlap:
            if pending is not None:
                _wgrad(pending[:6], 0)  # the first layer's weight gradients: nothing left to hide them under
            main.wait_stream(side)  # every gradient is complete before autograd hands them out
        if sync is not None:
            sync.wait()             # the collectives are joined on the main stream
        del keep
        ctx.ws = None
        return (None, grad_x, None) + tuple(grads.get(p) for p in ctx.param_list)


class CTC_Model(nn.Module):
    def __init__(self, add_cnn=False, cnn_param=None, rnn_param=None, num_class=39, drop_out=0.1):
        """
        add_cnn   [bool]:  put the Conv2d front before the RNN stack
        cnn_param [dict]:  {"layer": [[(cin, cout), (kh, kw), (sh, sw), (ph, pw), pool], ...],
                            "batch_norm": bool, "activate_function": nn.ReLU}
        rnn_param [dict]:  {"rnn_input_size", "rnn_hidden_size", "rnn_layers", "rnn_type", "bidirectional",
                            "batch_norm"}
        num_class  [int]:  number of output classes including blank
        drop_out [float]:  dropout probability used everywhere
        """
        super(CTC_Model, self).__init__()
        self.add_cnn = add_cnn
        self.cnn_param = cnn_param
        if rnn_param is None or type(rnn_param) != dict:
            raise ValueError("rnn_param need to be a dict to contain all params of rnn!")
        self.rnn_param = rnn_param
        self.num_class = num_class
        self.num_directions = 2 if rnn_param["bidirectional"] else 1
        self.drop_out = drop_out
        self.batch_tile = 0  # 0 = let the library pick the recurrent kernels' batch tile (16 or 32)
        self.overlap_wgrad = True  # weight-gradient GEMMs on a side stream, on the SMs the BPTT kernels leave idle
        self.overlap_gx = True     # input projection streamed chunk by chunk under the forward recurrence (_gx_stream_plan)
        self.gx_chunks = 8
        self.overlap_dg = True     # input-gradient / first-layer weight-gradient GEMMs follow the BPTT kernel chunk by chunk
        self.dg_chunks = 8
        # operand mode of every contraction: "bf16" (fast; gradients within ~1 % of fp32) or "x3" (split bf16 hi+lo, three
        # tensor-core products per contraction: gradients within 1e-3 of the reference's fp32 arithmetic)
        self.precision = os.environ.get("CTCB200_PRECISION", "bf16")
        self.grad_sync = None     # data parallel: a dist.GradSync whose per-layer all-reduces run inside backward()
        self.mask_source = None   # tests: callable(shape, p, device) -> keep-mask, replaces torch.rand for the dropout masks

        rnn_input_size = rnn_param["rnn_input_size"]
        if add_cnn:
            blocks = []
            out_channel = 1
            for n, spec in enumerate(cnn_param["layer"]):
                (in_channel, out_channel), kernel_size, stride, padding, pooling_size = spec
                blocks.append(("%d" % n, LayerCNN(in_channel, out_channel, kernel_size, stride, padding, pooling_size,
                                                  activation_function=cnn_param["activate_function"],
                                                  batch_norm=cnn_param["batch_norm"], dropout=drop_out)))
                try:
                    rnn_input_size = int(math.floor((rnn_input_size + 2 * padding[1] - kernel_size[1]) / stride[1]) + 1)
                except Exception:
                    pass  # 1-d convolution keeps the feature size
            self.conv = nn.Sequential(OrderedDict(blocks))
            rnn_input_size *= out_channel

        hidden = rnn_param["rnn_hidden_size"]
        stack = [("0", BatchRNN(input_size=rnn_input_size, hidden_size=hidden, rnn_type=rnn_param["rnn_type"],
                                bidirectional=rnn_param["bidirectional"], dropout=drop_out, batch_norm=False))]
        for i in range(rnn_param["rnn_layers"] - 1):
            stack.append(("%d" % (i + 1),
                          BatchRNN(input_size=self.num_directions * hidden, hidden_size=hidden,
                                   rnn_type=rnn_param["rnn_type"], bidirectional=rnn_param["bidirectional"],
                                   dropout=drop_out, batch_norm=rnn_param["batch_norm"])))
        self.rnns = nn.Sequential(OrderedDict(stack))

        if rnn_param["batch_norm"]:
            self.fc = nn.Sequential(nn.BatchNorm1d(self.num_directions * hidden),
                                    nn.Linear(self.num_directions * hidden, num_class, bias=False))
        else:
            self.fc = nn.Linear(self.num_directions * hidden, num_class, bias=False)
        self.log_softmax = nn.LogSoftmax(dim=-1)

    # -- checks that keep the CUDA path honest -------------------------------------------------------
    def _check_supported(self, x):
        _lib.require_cuda(x)
        if self.rnn_param["rnn_type"] not in (nn.LSTM, nn.GRU, nn.RNN):
            raise RuntimeError("the B200 path implements nn.LSTM / nn.GRU / nn.RNN layers (got %r)" % (self.rnn_param["rnn_type"],))
        if next(self.parameters()).device != x.device:
            raise RuntimeError("model parameters and input must live on the same CUDA device")
        if self.precision not in ("bf16", "x3"):
            raise RuntimeError("CTC_Model.precision must be 'bf16' or 'x3' (got %r)" % (self.precision,))
        check_hidden(self.rnn_param["rnn_hidden_size"], self.precision == "x3")

    def _rnn_params(self):
        plist = []
        for layer in self.rnns.children():
            if layer.batch_norm is not None:
                plist += [layer.batch_norm.weight, layer.batch_norm.bias]
            plist += [layer.rnn.weight_ih_l0, layer.rnn.weight_hh_l0]
            if self.num_directions == 2:
                plist += [layer.rnn.weight_ih_l0_reverse, layer.rnn.weight_hh_l0_reverse]
        if isinstance(self.fc, nn.Sequential):
            plist += [self.fc[0].weight, self.fc[0].bias, self.fc[1].weight]
        else:
            plist += [self.fc.weight]
        return plist

    def forward(self, x, visualize=False):
        # x: [batch, max_seq_length, feat_size]
        self._check_supported(x)
        with torch.cuda.device(x.device):   # launches, streams and the library's per-device state follow the tensors
            return self._forward(x, visualize)

    def _forward(self, x, visualize):
        visual = [x] if visualize else None
        # activations for BPTT are kept whenever a backward pass can follow (train or eval mode alike: eval only freezes
        # the BatchNorm statistics and disables dropout)
        need_grad = torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in self.parameters()))
        if self.add_cnn:
            from . import cnn
            seq = cnn.conv_front(self, x, need_grad)  # [N, T', Cc*F'] f32, feature index c*F' + f
            Nb, Tp, Dp = seq.shape
            if visualize:
                visual.append(seq)
                visual.append(seq.transpose(0, 1))
            src, geom = seq, (Tp, Nb, Dp, Dp, Tp * Dp, need_grad)
        else:
            if x.dtype != torch.float32:
                x = x.float()
            x = x.contiguous()
            Nb, Tp, Fp = x.shape
            src, geom = x, (Tp, Nb, Fp, Fp, Tp * Fp, need_grad)
        out = _RnnStackFn.apply(self, src, geom, *self._rnn_params())
        if visualize:
            visual.append(out)
            return out, visual
        return out

    # -- host-side helpers mirrored from the reference -------------------------------------------------
    def compute_wer(self, index, input_sizes, targets, target_sizes):
        """(edit-distance errors, reference tokens) over a batch of frame arg-max rows (model_ctc.py:187-202)."""
        from .decoder import collapse_frames, edit_distance
        batch_errs = 0
        batch_tokens = 0
        for i in range(len(index)):
            label = [int(v) for v in targets[i][:int(target_sizes[i])]]
            pred = collapse_frames(index[i][:int(input_sizes[i])], blank=0)
            batch_errs += edit_distance(label, pred)
            batch_tokens += len(label)
        return batch_errs, batch_tokens

    def compute_wer_device(self, log_probs, input_sizes, targets, target_sizes):
        """Same two numbers as compute_wer(torch.max(out, -1)[1].transpose(0, 1), ...) (train_ctc.py:51-52), computed on the
        device from the log-probabilities: arg-max + collapse + batched Levenshtein, one small D2H read at the end."""
        _, labels, lens = ops.greedy_decode(log_probs, input_sizes, blank=0)
        tsz = torch.as_tensor(target_sizes).to(device=log_probs.device, dtype=torch.int64)
        dist = ops.edit_distance(labels, lens, torch.as_tensor(targets).to(log_probs.device), tsz)
        both = torch.stack([dist.sum().to(torch.int64), tsz.sum()]).cpu()
        return int(both[0]), int(both[1])

    def add_weights_noise(self):
        # the reference's version rebinds a local and therefore changes nothing (model_ctc.py:204-207)
        return None

    @staticmethod
    def save_package(model, optimizer=None, decoder=None, epoch=None, loss_results=None, dev_loss_results=None,
                     dev_cer_results=None):
        package = {
            "rnn_param": model.rnn_param,
            "add_cnn": model.add_cnn,
            "cnn_param": model.cnn_param,
            "num_class": model.num_class,
            "_drop_out": model.drop_out,
            "state_dict": model.state_dict(),
        }
        if optimizer is not None:
            package["optim_dict"] = optimizer.state_dict()
        if decoder is not None:
            package["decoder"] = decoder
        if epoch is not None:
            package["epoch"] = epoch
        if loss_results is not None:
            package["loss_results"] = loss_results
            package["dev_loss_results"] = dev_loss_results
            package["dev_cer_results"] = dev_cer_results
        return package
