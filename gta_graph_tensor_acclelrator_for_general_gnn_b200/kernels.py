"""Thin Python wrappers over the compute entry points of libgta_b200.so.

One function per ISA instruction kind (SURVEY.md section 2.2): argument checking that needs
tensor metadata happens here, everything else in the C library.  Tensors are fp32, CUDA,
row-major with a row pitch that is a multiple of 4 elements (``alloc_table``).
"""
from __future__ import annotations

import torch

from . import _cabi
from .graph import DeviceGraph, Schedule, _require_cuda, _stream

LEAKY_SLOPE = 0.2

#: when a list, every wrapper below appends (name, start_event, end_event) recorded on the
#: current stream -- bench.py uses it to time the dominant kernel inside the timed region
EVENT_LOG = None


def _timed(name):
    def deco(fn):
        def wrapper(*a, **kw):
            log = EVENT_LOG
            if log is None:
                return fn(*a, **kw)
            start = torch.cuda.Event(enable_timing=True)
            end = torch.cuda.Event(enable_timing=True)
            start.record()
            out = fn(*a, **kw)
            end.record()
            log.append((name, start, end))
            return out
        wrapper.__name__ = fn.__name__
        wrapper.__doc__ = fn.__doc__
        return wrapper
    return deco


def pad4(n: int) -> int:
    return (n + 3) // 4 * 4


def pad_row(n: int, dtype=torch.float32) -> int:
    """Row pitch in elements: whole 16-byte pieces (4 fp32, 8 bf16)."""
    per = 16 // torch.empty((), dtype=dtype).element_size()
    return (n + per - 1) // per * per


def alloc_table(rows: int, width: int, device, zero: bool = False, dtype=torch.float32) -> torch.Tensor:
    """[rows, width] view of a buffer whose row pitch is padded to 16 bytes (fp32, or bf16 in the bf16 storage mode)."""
    ld = pad_row(width, dtype)
    buf = (torch.zeros if zero else torch.empty)((max(rows, 1), ld), dtype=dtype, device=device)
    return buf[:rows, :width]


def to_table(x: torch.Tensor) -> torch.Tensor:
    """Return ``x`` if its layout is already legal, else a padded copy (pad columns zeroed)."""
    if x.dtype not in (torch.float32, torch.bfloat16):
        raise TypeError("fp32 tables (or bf16 in the bf16 storage mode) only")
    if x.dim() == 1:
        x = x[:, None]
    per = 16 // x.element_size()
    if x.stride(1) == 1 and x.stride(0) % per == 0 and x.data_ptr() % 16 == 0 and x.stride(0) >= x.shape[1]:
        return x
    t = alloc_table(x.shape[0], x.shape[1], x.device, zero=True, dtype=x.dtype)
    t.copy_(x)
    return t


def _ld(t: torch.Tensor) -> int:
    if t.dim() != 2 or t.stride(1) != 1:
        raise ValueError("expected a row-major 2-D table")
    return int(t.stride(0)) if t.shape[0] > 1 else max(int(t.stride(0)), int(t.shape[1]))


class _Workspace:
    """Scratch buffer (fp32 elements) per (device, stream), grown by replacement.

    A buffer that has been handed out is never freed: a CUDA graph captured earlier keeps the device
    pointer it saw (the chain state of the aggregation kernels, the hi/lo split of W), so a later,
    larger request must not return that memory to the caching allocator.  Keying by stream keeps
    concurrent ``execute()`` calls on different streams (pipeline.HostPipeline) off each other's
    chain state; calls on one stream are ordered and may share."""

    def __init__(self):
        self.live = {}
        self.retired = []

    def get(self, n: int, device):
        if n == 0:
            return None
        device = torch.device(device)
        key = (device, torch.cuda.current_stream(device).cuda_stream)
        buf = self.live.get(key)
        if buf is None or buf.numel() < n:
            if buf is not None:
                self.retired.append(buf)
            buf = torch.empty(n, dtype=torch.float32, device=device)
            self.live[key] = buf
        return buf


_gemm_ws = _Workspace()
_agg_ws = _Workspace()      # chain state (partials + flags) of gta_aggregate_f32


def _chain_state(ws: _Workspace, num_slots: int, stride: int, f: int, device):
    """(partials, chain_state) pointers inside one workspace: num_slots*stride floats, then per 128-feature
    window num_slots int32 chain flags, then one int32 item counter per window and the slot-arrival counters
    of an exchange (always present)."""
    windows = (f + 127) // 128
    base = (num_slots * stride + 3) // 4 * 4
    buf = ws.get(base + (num_slots + 1) * windows + _cabi.MAX_RANKS, device)
    return (buf.data_ptr() if num_slots else None), buf.data_ptr() + 4 * base


def set_gemm_mode(mode: str) -> None:
    """'auto' (tcgen05 3xTF32 when eligible), 'simt' (FFMA) or 'tc' (tcgen05 or error)."""
    _cabi.check(_cabi.load().gta_gemm_set_mode({"auto": 0, "simt": 1, "tc": 2}[mode]), "gta_gemm_set_mode")


@_timed("gta_gemm_f32")
def gemm(x: torch.Tensor, w: torch.Tensor, al: torch.Tensor | None = None, ar: torch.Tensor | None = None,
         out: torch.Tensor | None = None, er_out: torch.Tensor | None = None, z_dtype=torch.float32):
    """COMP_MM applynode: ``Z = X.W`` and optionally the fused GAT ops 1/2 ``el = Z.Al``,
    ``er = Z.Ar``.  Returns ``Z`` or ``(Z, el, er)``.  ``out`` / ``er_out`` may be (strided) views of a
    larger table, e.g. this rank's slot of the gathered ``[F | H]`` source table.  ``z_dtype=torch.bfloat16``
    (bf16 storage mode) rounds Z once in the epilogue; el / er come from the fp32 accumulators."""
    lib = _cabi.load()
    _require_cuda(x, w, al, ar)
    n, k = x.shape
    k2, f = w.shape
    if k != k2:
        raise ValueError(f"X is [{n},{k}] but W is [{k2},{f}]")
    w = w.contiguous()
    z = out if out is not None else alloc_table(n, f, x.device, dtype=z_dtype)
    if z.dtype not in (torch.float32, torch.bfloat16):
        raise TypeError("Z is fp32 or bf16")
    heads = 0
    el = er = None
    if al is not None or ar is not None:
        heads = int((al if al is not None else ar).shape[1])
        if al is not None:      # el/er are dense [N,H]
            al = al.contiguous()
            el = torch.empty((n, heads), dtype=torch.float32, device=x.device)
        if ar is not None:
            ar = ar.contiguous()
            er = er_out if er_out is not None else torch.empty((n, heads), dtype=torch.float32, device=x.device)
            if er.stride(1) != 1 or er.shape != (n, heads):
                raise ValueError("er_out must be an [N, H] view with unit column stride")
    ws_bytes = int(lib.gta_gemm_workspace(k, f))
    ws = _gemm_ws.get((ws_bytes + 3) // 4, x.device)
    fn, name = (lib.gta_gemm_f32, "gta_gemm_f32") if z.dtype == torch.float32 else (lib.gta_gemm_f32_zbf16, "gta_gemm_f32_zbf16")
    _cabi.check(fn(_cabi.ptr(x), _ld(x), _cabi.ptr(w), f, _cabi.ptr(z), _ld(z), n, k, f,
                   _cabi.ptr(al), _cabi.ptr(ar), heads, _cabi.ptr(el), _cabi.ptr(er),
                   (int(er.stride(0)) if er is not None and n > 1 else heads), _cabi.ptr(ws), ws_bytes, _stream()), name)
    if al is None and ar is None:
        return z
    return z, el, er


#: below this many edges per work item a long list is walked with static striding (GTA_PHASE_STATIC)
STATIC_ITEM_EDGES = 48
STATIC_MIN_ITEMS = 1 << 18


def _launch_blocks(launch, sched: Schedule, block_events, num_edges: int = 0):
    """One launch for everything, or -- when the gathered table arrives chunk by chunk -- the first column
    block as soon as its chunk has landed and the rest after the last event."""
    if block_events is None:
        tiny = sched.num_items >= STATIC_MIN_ITEMS and num_edges < STATIC_ITEM_EDGES * sched.num_items
        launch(0, sched.num_items, _cabi.PHASE_ALL | (_cabi.PHASE_STATIC if tiny else 0))
        return
    if len(block_events) != sched.num_blocks:
        raise ValueError(f"{len(block_events)} chunk events for {sched.num_blocks} column blocks")
    # Two launches, not one per block: column block 0 starts as soon as its chunk has landed and
    # hides the transfer of all later chunks; the rest runs as ONE launch after the last event
    # (every extra launch boundary drains the SMs: measured 0.1 ms per boundary on the Reddit shape).
    # Chains of multi-item rows cross the boundary: the flags are cleared once, before the first launch.
    stream = torch.cuda.current_stream()
    nb = sched.num_blocks
    if block_events[0] is not None:
        stream.wait_event(block_events[0])
    first, last = sched.block_begin[0], sched.block_begin[1]
    launch(first, last - first, _cabi.PHASE_ALL)
    if nb > 1:
        if block_events[nb - 1] is not None:
            stream.wait_event(block_events[nb - 1])      # chunks complete in order on the communication stream
        first, last = sched.block_begin[1], sched.block_begin[nb]
        if last > first:
            launch(first, last - first, _cabi.PHASE_MAIN)


@_timed("gta_aggregate_f32")
def aggregate(g: DeviceGraph, x: torch.Tensor, w: torch.Tensor | None = None, rowden: torch.Tensor | None = None,
              epilogue: int = _cabi.EPI_NONE, sched: Schedule | None = None, out: torch.Tensor | None = None,
              block_events=None, exchange=None):
    """COMP_MUL_COMP_ADD / COMP_ADD gather: ``out[i] = epi(sum_k w[k] (x) x[src k])``;
    with ``rowden`` the weight is ``w[k,h] / rowden[i,h]`` (GAT op 9).  ``block_events[b]`` (optional)
    is the CUDA event after which column block b of the gathered table is valid.  ``exchange`` (a
    ``dist.Gate``): ``x`` is this step's gathered table of a fused exchange and the launch pulls the peers' slots
    itself; the work list is then cut at the slot boundaries."""
    lib = _cabi.load()
    _require_cuda(x, w, rowden)
    if exchange is not None:
        sched = g.schedule(col_cuts=exchange.block_cuts)
    sched = sched or g.schedule_for(_ld(x) * x.element_size())
    f = int(x.shape[1])
    rows = sched.row_end - sched.row_begin
    o = out if out is not None else alloc_table(rows, f, x.device)
    if f % 4 and _ld(x) >= pad4(f) and _ld(o) >= pad4(f):
        f = pad4(f)      # whole 4-feature pieces: run over the pad columns too (independent columns, never read back)
    fn, fname = (lib.gta_aggregate_f32, "gta_aggregate_f32") if x.dtype == torch.float32 else \
        (lib.gta_aggregate_bf16, "gta_aggregate_bf16")
    wmode, wh = _cabi.W_NONE, 0
    if w is not None:
        if w.dim() == 1:
            w = w[:, None]
        w = w.contiguous()
        wh = int(w.shape[1])
        wmode = _cabi.W_EDGE_DIV if rowden is not None else _cabi.W_EDGE
        if rowden is not None:
            rowden = rowden.contiguous()
    partials, chain = _chain_state(_agg_ws, sched.num_slots, f, f, x.device)

    def launch(first, count, phases):
        _cabi.check(fn(sched.items.data_ptr() + 16 * first, count, _cabi.ptr(sched.row_slots),
                       sched.num_slots, _cabi.ptr(g.indices), wmode, _cabi.ptr(w), wh,
                       _cabi.ptr(rowden), _cabi.ptr(x), _ld(x), _cabi.ptr(o), _ld(o), f, epilogue,
                       partials, chain, exchange.byref() if exchange is not None else None,
                       phases, _stream()), fname)
    _launch_blocks(launch, sched, block_events, g.num_edges)
    return o


@_timed("gta_aggregate_edge_sum_f32")
def aggregate_edge_sum(g: DeviceGraph, edge: torch.Tensor | None = None, x: torch.Tensor | None = None,
                       rowterm: torch.Tensor | None = None, unary: int = _cabi.UN_COPY, slope: float = LEAKY_SLOPE,
                       epilogue: int = _cabi.EPI_NONE, sched: Schedule | None = None):
    """``out[i] = epi(sum_k unary(edge[k] + x[src k] + rowterm[i]))`` in one pass (PNA ops 5-8): ``edge`` [E, F] in
    CSR edge order, ``x`` [sources, F] gathered by source, ``rowterm`` [N, F]; any may be None (not all).  fp32
    tables (``to_table``); nothing E x F is written."""
    lib = _cabi.load()
    given = [t for t in (edge, x, rowterm) if t is not None]
    if not given:
        raise ValueError("aggregate_edge_sum: at least one of edge / x / rowterm")
    _require_cuda(*given)
    f = int(given[0].shape[1])
    if any(int(t.shape[1]) != f or t.dtype != torch.float32 for t in given):
        raise ValueError("aggregate_edge_sum: fp32 operands of one width")
    sched = sched or (g.schedule_for(_ld(x) * 4) if x is not None else g.schedule())
    rows = sched.row_end - sched.row_begin
    o = alloc_table(rows, f, given[0].device)
    if f % 4 and all(_ld(t) >= pad_row(f, torch.float32) for t in given + [o]):
        f = pad_row(f, torch.float32)      # run over the pad columns too (independent columns, never read back)
    partials, chain = _chain_state(_agg_ws, sched.num_slots, f, f, o.device)

    def launch(first, count, phases):
        _cabi.check(lib.gta_aggregate_edge_sum_f32(
            sched.items.data_ptr() + 16 * first, count, _cabi.ptr(sched.row_slots), sched.num_slots, _cabi.ptr(g.indices),
            _cabi.ptr(edge), _ld(edge) if edge is not None else 0, _cabi.ptr(x), _ld(x) if x is not None else 0,
            _cabi.ptr(rowterm), _ld(rowterm) if rowterm is not None else 0, unary, slope, _cabi.ptr(o), _ld(o), f,
            epilogue, partials, chain, phases, _stream()), "gta_aggregate_edge_sum_f32")
    _launch_blocks(launch, sched, None, g.num_edges)
    return o


_gat_ws = _Workspace()      # chain state of the single-pass GAT kernel


def gather_peak(table_bytes: int = 40 << 20, f: int = 128, gathers_per_group: int = 4096, iters: int = 5) -> dict:
    """Measured ceiling of the gather kernels on this device (``gta_gather_peak_probe``): random whole-row gathers
    from an L2-resident table with the kernels' own load instruction.  Returns ``{"gbs": ..., "rows": ..., ...}``."""
    lib = _cabi.load()
    dev = torch.device("cuda", torch.cuda.current_device())
    rows = max(table_bytes // (f * 4), 1)
    table = alloc_table(rows, f, dev)
    table.normal_()
    sink = torch.zeros(1 << 20, dtype=torch.float32, device=dev)
    groups = 0
    times = []
    for it in range(iters + 2):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        groups = int(lib.gta_gather_peak_probe(_cabi.ptr(table), rows, _ld(table), f, gathers_per_group, _cabi.ptr(sink),
                                               _stream()))
        b.record()
        if groups <= 0:
            _cabi.check(-groups, "gta_gather_peak_probe")
        b.synchronize()
        if it >= 2:
            times.append(a.elapsed_time(b))
    ms = min(times)
    byts = groups * gathers_per_group * f * 4
    return {"gbs": byts / (ms * 1e-3) / 1e9, "ms": ms, "rows": rows, "row_bytes": f * 4, "table_mb": rows * f * 4 / 2**20,
            "gathers": groups * gathers_per_group, "how": "gta_gather_peak_probe: best of %d launches" % iters}


def er_stats(er: torch.Tensor, col_block: int = 0) -> torch.Tensor | None:
    """Ordered-int codes of ``max er`` / ``max -er`` per column block and head (``gta_er_stats``), or None
    when the head count is not a power of two (the aggregation then runs the online softmax)."""
    lib = _cabi.load()
    n, heads = int(er.shape[0]), int(er.shape[1])
    if heads < 1 or heads > 32 or heads & (heads - 1):
        return None
    n_cb = int(lib.gta_schedule_col_blocks(n, col_block))
    stats = torch.empty((n_cb, 2, heads), dtype=torch.int32, device=er.device)
    lder = int(er.stride(0)) if n > 1 else max(int(er.stride(0)), heads)
    _cabi.check(lib.gta_er_stats(_cabi.ptr(er), lder, n, col_block if n_cb > 1 else 0, heads, _cabi.ptr(stats),
                                 _stream()), "gta_er_stats")
    return stats


@_timed("gta_gat_aggregate_f32")
def gat_aggregate(g: DeviceGraph, el: torch.Tensor, er: torch.Tensor, z: torch.Tensor, slope: float = LEAKY_SLOPE,
                  epilogue: int = _cabi.EPI_ELU, sched: Schedule | None = None, out: torch.Tensor | None = None,
                  want_stats: bool = False, block_events=None, bounded: bool = True, exchange=None):
    """GAT ops 3-13 in one pass: returns ``out`` or ``(out, rowmax, rowsum)``.  ``bounded`` shifts the softmax
    by the per-(row, column block) bound ``leaky(el + max er)`` where the block's er range allows it (see
    ``gta_er_stats``); ``want_stats`` runs the online softmax with a running maximum, and so does ``False`` without
    an exchange.  ``exchange`` (a ``dist.Gate``): ``z`` / ``er`` are views of this step's gathered table of a fused
    exchange, see ``aggregate``; the bound then comes from the er ranges the slot owners published with the step,
    whatever ``bounded`` says, so only ``want_stats`` selects the online softmax there."""
    lib = _cabi.load()
    _require_cuda(el, er, z)
    if exchange is not None:
        sched = g.schedule(col_cuts=exchange.block_cuts)
    sched = sched or g.schedule_for(_ld(z) * z.element_size())
    f = int(z.shape[1])
    heads = int(el.shape[1])
    rows = sched.row_end - sched.row_begin
    el = el.contiguous()
    if er.stride(1) != 1 or er.data_ptr() % 16 or (er.stride(0) % 4 and heads % 4 == 0):
        er = er.contiguous()     # a strided view (er living beside z in one gathered table) is used in place
    lder = int(er.stride(0)) if er.shape[0] > 1 else max(int(er.stride(0)), heads)
    o = out if out is not None else alloc_table(rows, f, z.device)
    rowmax = rowsum = None
    if want_stats:
        rowmax = torch.empty((rows, heads), dtype=torch.float32, device=z.device)
        rowsum = torch.empty((rows, heads), dtype=torch.float32, device=z.device)
    stride = int(lib.gta_gat_partial_stride(f, heads))
    partials, chain = _chain_state(_gat_ws, sched.num_slots, stride, f, z.device)
    col_block = sched.col_block if sched.num_blocks > 1 else 0
    # with chunk events the table is still arriving: its er range is not known before the launch
    # (with an exchange the slot owners publish their er range and the kernel reads it from the signal block);
    # an empty work list (a rank without rows) launches nothing at all
    stats = er_stats(er, col_block) if (bounded and not want_stats and block_events is None and exchange is None
                                        and sched.num_items > 0) else None

    fn, fname = (lib.gta_gat_aggregate_f32, "gta_gat_aggregate_f32") if z.dtype == torch.float32 else \
        (lib.gta_gat_aggregate_bf16, "gta_gat_aggregate_bf16")

    def launch(first, count, phases):
        _cabi.check(fn(sched.items.data_ptr() + 16 * first, count, _cabi.ptr(sched.row_slots),
                       sched.num_slots, _cabi.ptr(g.indices), _cabi.ptr(el),
                       _cabi.ptr(er), lder, heads, slope, _cabi.ptr(z), _ld(z), _cabi.ptr(o),
                       _ld(o), f, epilogue, _cabi.ptr(rowmax), _cabi.ptr(rowsum),
                       partials, chain, _cabi.ptr(stats), col_block,
                       exchange.byref() if exchange is not None else None, phases, _stream()), fname)
    _launch_blocks(launch, sched, block_events, g.num_edges)
    if want_stats:
        return o, rowmax, rowsum
    return o


@_timed("gta_gat_logits_f32")
def gat_logits(g: DeviceGraph, el: torch.Tensor, er: torch.Tensor, slope: float = LEAKY_SLOPE,
               stabilize: bool = True):
    """GAT block [4,5,6,7,8]: returns ``(p [E,H], rowmax [N,H], rowsum [N,H])``."""
    lib = _cabi.load()
    _require_cuda(el, er)
    heads = int(el.shape[1])
    el = el.contiguous()
    er = er.contiguous()
    rows = g.num_rows
    p = torch.empty((max(g.num_edges, 1), heads), dtype=torch.float32, device=el.device)[:g.num_edges]
    rowmax = torch.empty((rows, heads), dtype=torch.float32, device=el.device)
    rowsum = torch.empty((rows, heads), dtype=torch.float32, device=el.device)
    _cabi.check(lib.gta_gat_logits_f32(_cabi.ptr(g.indptr), _cabi.ptr(g.indices), 0, rows, _cabi.ptr(el),
                                       _cabi.ptr(er), heads, slope, int(stabilize), _cabi.ptr(p), _cabi.ptr(rowmax),
                                       _cabi.ptr(rowsum), _stream()), "gta_gat_logits_f32")
    return p, rowmax, rowsum


def edge_binary(g: DeviceGraph, op: int, a: torch.Tensor, kind_a: int, b: torch.Tensor, kind_b: int):
    lib = _cabi.load()
    a = a if a.dim() == 2 else a[:, None]
    b = b if b.dim() == 2 else b[:, None]
    a, b = a.contiguous(), b.contiguous()
    wo = max(int(a.shape[1]), int(b.shape[1]))
    out = torch.empty((max(g.num_edges, 1), wo), dtype=torch.float32, device=a.device)[:g.num_edges]
    _cabi.check(lib.gta_edge_binary_f32(_cabi.ptr(g.indptr), _cabi.ptr(g.indices), 0, g.num_rows, op,
                                        _cabi.ptr(a), kind_a, int(a.shape[1]), int(a.shape[1]),
                                        _cabi.ptr(b), kind_b, int(b.shape[1]), int(b.shape[1]),
                                        _cabi.ptr(out), wo, wo, _stream()), "gta_edge_binary_f32")
    return out


def edge_unary(g: DeviceGraph, op: int, a: torch.Tensor, kind_a: int, slope: float = LEAKY_SLOPE):
    lib = _cabi.load()
    a = a if a.dim() == 2 else a[:, None]
    a = a.contiguous()
    wa = int(a.shape[1])
    out = torch.empty((max(g.num_edges, 1), wa), dtype=torch.float32, device=a.device)[:g.num_edges]
    _cabi.check(lib.gta_edge_unary_f32(_cabi.ptr(g.indptr), _cabi.ptr(g.indices), 0, g.num_rows, op, slope,
                                       _cabi.ptr(a), kind_a, wa, wa, _cabi.ptr(out), wa, _stream()),
                "gta_edge_unary_f32")
    return out


def node_binary(op: int, a: torch.Tensor, b: torch.Tensor):
    lib = _cabi.load()
    a = a if a.dim() == 2 else a[:, None]
    b = b if b.dim() == 2 else b[:, None]
    wo = max(int(a.shape[1]), int(b.shape[1]))
    n = int(a.shape[0])
    out = alloc_table(n, wo, a.device)
    _cabi.check(lib.gta_node_binary_f32(op, _cabi.ptr(a), int(a.shape[1]), _ld(a), _cabi.ptr(b), int(b.shape[1]),
                                        _ld(b), _cabi.ptr(out), wo, _ld(out), n, _stream()), "gta_node_binary_f32")
    return out


def node_unary(op: int, a: torch.Tensor, slope: float = LEAKY_SLOPE):
    lib = _cabi.load()
    a = a if a.dim() == 2 else a[:, None]
    n, w = int(a.shape[0]), int(a.shape[1])
    out = alloc_table(n, w, a.device)
    _cabi.check(lib.gta_node_unary_f32(op, slope, _cabi.ptr(a), _ld(a), _cabi.ptr(out), _ld(out), w, n, _stream()),
                "gta_node_unary_f32")
    return out
