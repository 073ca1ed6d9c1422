"""The fused exchange (dist.FusedExchange, csrc/exchange.cuh) with every rank emulated on ONE GPU, held to the fp64
oracle step by step, with different data at every step.

In an exchange the first copy_ctas CTAs of the aggregation launch pull the peers' slots into the rank's gathered table
while the other CTAs wait at the slot gates, and the GAT kernels take their softmax bound from the er ranges the peers
publish into stats[step & 1] of the signal block.  A slot that is never copied, a swapped table parity or statistics
of the wrong step or slot all leave values of an EARLIER step behind: only data that changes from step to step, and er
offsets far enough apart that a stale bound overflows or underflows exp, make such a fault visible.

Every compiled aggregate and GAT instance (the case table of test_gpu_instances.py) runs through a world-4 exchange,
whose slot groups [[0], [1], [2, 3]] give items that span two slots; then the partition edges (world sizes, one copy
CTA, ranks without rows, 3 and 32 heads, a wide er range beside narrow ones); then static striding on widths that
need a second feature window.  (Real ranks, one GPU each: test_gpu_multiprocess.py.)
"""
import types
import zlib

import numpy as np
import pytest

from conftest import assert_close_rowscale
from oracle import gta_oracle as O
from gta_graph_tensor_acclelrator_for_general_gnn_b200 import _cabi, synthetic
from test_gpu_bf16 import _bf16_round
from test_gpu_instances import CASES, _case_id, _inputs, crafted_graph, launched
from test_gpu_kernels import _gat_from_z

pytestmark = pytest.mark.gpu


# ---- the emulated exchange and one step of it ------------------------------------------------------------------------
def emulated(full, world, copy_ctas=0):
    """Partitions and FusedExchange objects of every rank of ``world``, all on this GPU."""
    from gta_graph_tensor_acclelrator_for_general_gnn_b200 import dist as gdist
    parts = [gdist.make_partition(full, r, world) for r in range(world)]
    exs = [gdist.FusedExchange(p, copy_ctas=copy_ctas) for p in parts]
    for ex in exs:
        ex.emulate_with(exs)
    return parts, exs


def release(exs):
    """Free the IPC tables and signal blocks of emulated exchanges (nothing of them is used afterwards)."""
    import torch
    torch.cuda.synchronize()
    for ex in exs:
        for st in ex._state.values():
            for buf in st["tables"] + [st["signals"]]:
                buf.close()


def run_step(parts, exs, produce, consume):
    """One emulated step.  ``produce(p, ex) -> (tables, gate, *args)`` writes rank p's slot and publishes it
    (gta_exchange_publish); it runs on EVERY rank before any rank's ``consume(p, tables, gate, *args)`` launches its
    aggregation -- a launch whose peers have not all published spins in its copy CTAs until the bounded wait traps.
    ``tables`` is the tuple of the rank's gathered-table views.  Returns ``[(output, tables, gate)]`` in rank order."""
    import torch
    staged = [produce(p, ex) for p, ex in zip(parts, exs)]
    outs = [consume(p, *s) for p, s in zip(parts, staged)]
    torch.cuda.synchronize()
    return [(o, s[0], s[1]) for o, s in zip(outs, staged)]


def assert_slots_hold(parts, results, wants, what):
    """After the launch, every slot of every rank's table holds its owner's rows OF THIS STEP: ``wants`` are the whole
    step's source tensors (device, the tables' dtypes) in the order of each rank's ``tables``.  A rank without rows has
    no items and launches nothing, so it pulls nothing."""
    import torch
    for p, (_, tables, _) in zip(parts, results):
        if p.rows == 0:
            continue
        for k in range(p.world):
            q = p.owner_of(k)
            b0, b1 = p.bounds[q], p.bounds[q + 1]
            for t, want in zip(tables, wants):
                assert torch.equal(t[k * p.stride: k * p.stride + b1 - b0], want[b0:b1]), \
                    f"{what}: slot {k} of rank {p.rank} does not hold rank {q}'s rows of this step"


def _cat(results, pick=lambda o: o):
    import torch
    return torch.cat([pick(o) for o, _, _ in results])


def _owner_of_rows(bounds, n):
    return (np.searchsorted(np.asarray(bounds), np.arange(n), side="right") - 1).astype(np.int64)


# ---- er offsets that make stale statistics fail ------------------------------------------------------------------------
# Data set d of a step shifts the er of owner q by ER_OFFSET[d](q) around N(0, 1): a bound taken from the statistics of
# another step (d0 -> d1: +100, d1 -> d2: -100 for half the owners) or of a neighbouring slot inside d2 then overflows
# or underflows exp instead of being silently right.  |el + er| stays below 128, where half an fp32 ulp is 3.8e-6.
ER_OFFSET = {0: lambda q: 0.0, 1: lambda q: 100.0, 2: lambda q: 100.0 if q % 2 else -100.0}


def _er_offsets(d, owner):
    return np.array([ER_OFFSET[d](q) for q in range(int(owner.max()) + 1)], np.float32)[owner][:, None]


def _stale_bound_breaks(indptr, indices, owner, el, er, stale_hi):
    """In fp32, exp(e - stale bound) is inf or 0 for some edge: e = leaky(el[i] + er[j]) and the stale bound is
    leaky(el[i] + stale_hi[owner(j)]), stale_hi [ranks, heads] the per-owner er maximum the kernel would have read."""
    rows = O.row_ids(indptr)
    e = O.leaky_relu(el[rows] + er[indices])
    b = O.leaky_relu(el[rows] + stale_hi[owner[indices]])
    with np.errstate(over="ignore", under="ignore"):
        p = np.exp(e - b)
    return bool(np.any(np.isinf(p) | (p == 0)))


def _er_max_per_owner(er, owner, world):
    return np.stack([er[owner == q].max(axis=0) if np.any(owner == q) else np.full(er.shape[1], -np.inf, np.float32)
                     for q in range(world)]).astype(np.float32)


# ---- one GAT / aggregate step through the exchange, checked against the oracle ------------------------------------------
def _gat_step(H, parts, exs, z, el, er, dtype, what, profile_instance=None):
    """Publish z / er of every rank, run the bounded (exchange statistics) and the want_stats (online) path, check slots,
    outputs, rowmax and rowsum against fp64.  Returns the concatenated (bounded, online) outputs."""
    import torch
    from gta_graph_tensor_acclelrator_for_general_gnn_b200 import kernels
    zd = torch.from_numpy(z).cuda()
    zd = zd.to(torch.bfloat16) if dtype == "bf16" else zd
    erd = torch.from_numpy(er).cuda()
    # el of each rank in an allocation of its own, as a rank's GEMM writes it: the kernel takes el 16-byte aligned
    els = [torch.from_numpy(np.ascontiguousarray(el[p.row_begin:p.row_end])).cuda() for p in parts]

    def produce(p, ex):
        zt, ert, gate = ex.gather_pair(zd[p.row_begin:p.row_end], erd[p.row_begin:p.row_end])
        return (zt, ert), gate

    def consume(p, tables, gate):
        zt, ert = tables
        e = els[p.rank]
        return (kernels.gat_aggregate(p.local, e, ert, zt, exchange=gate),
                kernels.gat_aggregate(p.local, e, ert, zt, exchange=gate, want_stats=True))

    if profile_instance is None:
        res = run_step(parts, exs, produce, consume)
    else:
        res, ran = launched(lambda: run_step(parts, exs, produce, consume))
        assert ran == {profile_instance}, f"{what}: launched {sorted(ran)}, not {profile_instance}"
    assert_slots_hold(parts, res, (zd, erd), what)
    r = _gat_from_z(H.indptr, H.indices, z, el, er)
    scale = O.gat_rowscale(H.indptr, H.indices, z.astype(np.float64), r["alpha"])
    bounded, online = _cat(res, lambda o: o[0]), _cat(res, lambda o: o[1][0])
    assert_close_rowscale(bounded.cpu().numpy(), r["Y"], scale, what=what + " bounded")
    assert_close_rowscale(online.cpu().numpy(), r["Y"], scale, what=what + " online")
    np.testing.assert_allclose(_cat(res, lambda o: o[1][1]).cpu().numpy(), r["rowmax"], rtol=1e-6, atol=1e-6,
                               err_msg=what + " rowmax")
    np.testing.assert_allclose(_cat(res, lambda o: o[1][2]).cpu().numpy(), r["S"], rtol=2e-5, err_msg=what + " rowsum")
    return bounded, online


def _aggregate_step(H, parts, exs, x, w, rowden, weff, dtype, what, profile_instance=None):
    """Publish x of every rank, aggregate with the edge weights permuted into each rank's edge order, check slots and
    output against fp64.  Returns the concatenated output."""
    import torch
    from gta_graph_tensor_acclelrator_for_general_gnn_b200 import kernels
    xd = torch.from_numpy(x).cuda()
    xd = xd.to(torch.bfloat16) if dtype == "bf16" else xd
    wd = None if w is None else torch.from_numpy(w).cuda()
    rd = None if rowden is None else torch.from_numpy(rowden).cuda()

    def produce(p, ex):
        table, gate = ex.gather_one(xd[p.row_begin:p.row_end])
        return (table,), gate

    def consume(p, tables, gate):
        e0, e1 = int(H.indptr[p.row_begin]), int(H.indptr[p.row_end])
        return kernels.aggregate(p.local, tables[0], None if wd is None else p.permute_edges(wd[e0:e1]),
                                 None if rd is None else rd[p.row_begin:p.row_end], exchange=gate)

    if profile_instance is None:
        res = run_step(parts, exs, produce, consume)
    else:
        res, ran = launched(lambda: run_step(parts, exs, produce, consume))
        assert ran == {profile_instance}, f"{what}: launched {sorted(ran)}, not {profile_instance}"
    assert_slots_hold(parts, res, (xd,), what)
    out = _cat(res)
    want = O.spmm(H.indptr, H.indices, weff, x)
    scale = O.spmm(H.indptr, H.indices, None if weff is None else np.abs(weff), np.abs(x))
    assert_close_rowscale(out.cpu().numpy(), want, scale, what=what)
    return out


def _host_graph(n, dst, src):
    from gta_graph_tensor_acclelrator_for_general_gnn_b200 import graph
    indptr, indices, _ = O.csr_build(dst, src, n)
    return types.SimpleNamespace(n=n, e=len(indices), indptr=indptr, indices=indices, rows=O.row_ids(indptr),
                                 full=graph.csr_from_coo(dst, src, n))


# ---- every aggregate and GAT instance through a world-4 exchange --------------------------------------------------------
#: data sets of the four steps: both table parities twice; step 4 overwrites the d1 of step 2 with d0
STEPS = (0, 1, 2, 0)
EXCHANGE_CASES = [(c, i) for c, i in CASES if c[0] in ("aggregate", "gat")]          # edge_sum has no exchange entry


@pytest.fixture(scope="module")
def W4():
    _cabi.load()
    H = _host_graph(*crafted_graph())
    from gta_graph_tensor_acclelrator_for_general_gnn_b200 import dist as gdist
    assert gdist.slot_groups(4) == [[0], [1], [2, 3]]
    H.parts, H.exs = emulated(H.full, 4)
    H.owner = _owner_of_rows(H.parts[0].bounds, H.n)
    yield H
    release(H.exs)


def _gat_data(call, d, owner, offsets=True):
    _, dtype, f, heads = call
    z = _inputs(call, f"z{d}", (len(owner), f))
    if dtype == "bf16":
        z = _bf16_round(z)
    el = _inputs(call, f"el{d}", (len(owner), heads))
    er = _inputs(call, f"er{d}", (len(owner), heads))
    if offsets:
        er = er + _er_offsets(d, owner)
    return z, el, er.astype(np.float32)


def _aggregate_data(H, call, d):
    _, dtype, f, wh, div = call
    x = _inputs(call, f"x{d}", (H.n, f))
    if dtype == "bf16":
        x = _bf16_round(x)          # the kernel sees exactly these values: fp32 tolerance
    w = rowden = weff = None
    if wh:
        w = np.random.default_rng(zlib.crc32(repr((call, "w", d)).encode())).uniform(0.1, 1.0, (H.e, wh)).astype(np.float32)
        weff = w.astype(np.float64)
        if div:
            rowden = O.segment_sum(weff, H.indptr).astype(np.float32)
            weff = weff / rowden[H.rows]
    return x, w, rowden, weff


@pytest.mark.parametrize("call,instance", EXCHANGE_CASES, ids=[_case_id(c) for c, _ in EXCHANGE_CASES])
def test_instance_through_exchange_step_by_step(W4, call, instance):
    """Four steps of changing data (d0 d1 d2 d0) through the world-4 exchange: per step the profiled instance, every
    rank's slots and the output against the oracle of THIS step's data; step 4 must repeat step 1 bit for bit."""
    outs = []
    for s, d in enumerate(STEPS):
        what = f"{_case_id(call)} step {s + 1} (d{d})"
        if call[0] == "gat":
            outs.append(_gat_step(W4, W4.parts, W4.exs, *_gat_data(call, d, W4.owner), call[1], what, instance))
        else:
            x, w, rowden, weff = _aggregate_data(W4, call, d)
            outs.append((_aggregate_step(W4, W4.parts, W4.exs, x, w, rowden, weff, call[1], what, instance),))
    for a, b in zip(outs[0], outs[3]):
        assert a.equal(b), f"{_case_id(call)}: step 4 (d0 again) differs from step 1"
    heads = call[3] if call[0] == "gat" else 0
    if heads and heads <= 32 and heads & (heads - 1) == 0:          # the bound path runs: stale statistics must show
        data = {d: _gat_data(call, d, W4.owner) for d in (0, 1, 2)}
        for prev, d in ((0, 1), (1, 2)):
            _, el, er = data[d]
            stale = _er_max_per_owner(data[prev][2], W4.owner, 4)
            assert _stale_bound_breaks(W4.indptr, W4.indices, W4.owner, el, er, stale), \
                f"{_case_id(call)}: a bound from d{prev}'s statistics would not break d{d}"
        _, el, er = data[2]
        hi = _er_max_per_owner(er, W4.owner, 4)
        assert _stale_bound_breaks(W4.indptr, W4.indices, W4.owner, el, er, np.roll(hi, 1, axis=0)), \
            f"{_case_id(call)}: a bound from the neighbouring slot's statistics would not break d2"


# ---- partition edges ------------------------------------------------------------------------------------------------------
def _hub_graph():
    """Three hub rows holding three quarters of the edges in front of a sparse power-law graph: the edge-balanced
    bounds of 8 ranks then leave some ranks without rows."""
    g = synthetic.powerlaw_graph(3000, 6000, seed=9, i0=3.0)
    n = g.num_nodes
    hubs = [np.delete(np.arange(n, dtype=np.int32), r) for r in range(3)]
    dst = np.concatenate([np.full(len(h), r, np.int32) for r, h in enumerate(hubs)] + [g.dst.astype(np.int32)])
    src = np.concatenate(hubs + [g.src.astype(np.int32)])
    return n, dst, src


#: (world, copy_ctas, graph, heads override, wide er slot)
EDGES = {
    "world2": (2, 0, "crafted", None, False),
    "world3": (3, 0, "crafted", None, False),
    "world5": (5, 0, "crafted", None, False),
    "world7": (7, 0, "crafted", None, False),
    "world8": (8, 0, "crafted", None, False),
    "world3-copy1": (3, 1, "crafted", None, False),
    "world5-copy1": (5, 1, "crafted", None, False),
    "world8-copy1": (8, 1, "crafted", None, False),
    "empty-ranks": (8, 0, "hub", None, False),
    "heads3": (4, 0, "crafted", 3, False),
    "heads32": (4, 0, "crafted", 32, False),
    "wide-er": (4, 0, "crafted", None, True),
}
EDGE_RUNS = [pytest.param(kind, v, id=f"{kind}-{v}")
             for kind in ("gat-f32", "gat-bf16", "gcn") for v in EDGES
             if not (kind != "gat-f32" and EDGES[v][3] is not None)          # bf16 GAT: 1, 2 or 4 heads; GCN: no heads
             and not (kind == "gcn" and EDGES[v][4])]


@pytest.fixture(scope="module")
def edge_graphs():
    _cabi.load()
    return {"crafted": _host_graph(*crafted_graph()), "hub": _host_graph(*_hub_graph())}


@pytest.mark.parametrize("kind,variant", EDGE_RUNS)
def test_exchange_partition_edges(edge_graphs, kind, variant):
    """Four steps of changing data (d0 d1 d2 d0) through the slot-group shapes of other world sizes (3: [[0],[1],[2]],
    5: [[0],[1],[2,3,4]], 7: [[0],[1,2],[3,4,5,6]]), a single copy CTA, ranks without rows (slots with valid_rows = 0),
    3 and 32 heads, and one slot whose er spans about +-300 beside narrow ones (items that touch it take the online
    softmax)."""
    world, copy_ctas, gname, heads_override, wide = EDGES[variant]
    H = edge_graphs[gname]
    parts, exs = emulated(H.full, world, copy_ctas)
    try:
        if gname == "hub":
            assert any(p.rows == 0 for p in parts), f"bounds {parts[0].bounds} leave every rank rows"
            assert sum(p.rows > 0 for p in parts) >= 2
        owner = _owner_of_rows(parts[0].bounds, H.n)
        outs = []
        for s, d in enumerate((0, 1, 2, 0)):
            what = f"{kind} {variant} step {s + 1} (d{d})"
            if kind == "gcn":
                x = _inputs(("gcn", variant), f"x{d}", (H.n, 64))
                ew = synthetic.gcn_edge_norm(H.indptr, H.indices)
                outs.append((_aggregate_step(H, parts, exs, x, ew[:, None], None, ew, "f32", what),))
                continue
            heads = heads_override or 4
            f = 96 if heads == 3 else 128
            call = ("gat", kind[4:], f, heads)
            z, el, er = _gat_data(call, d, owner, offsets=not wide)
            if wide:          # a different owner's slot spans about +-300 at every step; the others stay narrow
                er[owner == (1 + d) % world] *= 80.0
            outs.append(_gat_step(H, parts, exs, z, el, er, kind[4:], what))
        for a, b in zip(outs[0], outs[3]):
            assert a.equal(b), f"{kind} {variant}: step 4 (d0 again) differs from step 1"
    finally:
        release(exs)


# ---- static striding through an exchange, two feature windows ------------------------------------------------------------
#: widths just above one window (the tables stay small): (kind, f, heads or weight heads)
STATIC_WIDE = [("gat", 136, 2), ("gat", 144, 12), ("aggregate", 132, 3), ("aggregate", 260, 0)]


@pytest.fixture(scope="module")
def static_world2():
    import torch
    from gta_graph_tensor_acclelrator_for_general_gnn_b200 import dist as gdist, graph
    _cabi.load()
    g = synthetic.powerlaw_graph(800_000, 4_800_000, seed=5, i0=50.0, name="wide-low-degree")
    n = g.num_nodes
    full = graph.csr_from_coo(g.dst, g.src, n)
    parts, exs = emulated(full, 2)
    cuts = tuple((grp[-1] + 1) * parts[0].stride for grp in gdist.slot_groups(2)[:-1])
    for p in parts:          # 32 group-steps for every warp of 148 SMs x 64 resident warps: static whatever the occupancy
        assert p.local.schedule(col_cuts=cuts).num_items >= 32 * 148 * 64
    gen = torch.Generator(device="cuda").manual_seed(21)
    S = types.SimpleNamespace(
        n=n, full=full, parts=parts, exs=exs, indptr=full.indptr.cpu().numpy(), indices=full.indices.cpu().numpy(),
        z=torch.randn((n, 260), generator=gen, device="cuda"),
        el={h: torch.randn((n, h), generator=gen, device="cuda") for h in (2, 12)},
        er={h: torch.randn((n, h), generator=gen, device="cuda") for h in (2, 12)},
        w=torch.rand((full.num_edges, 3), generator=gen, device="cuda") + 0.1)
    yield S
    release(exs)


def _sample_oracle(S, kind, f, h, rows):
    """fp64 oracle of the sampled destination rows only (the whole graph is too large for the host)."""
    deg = np.diff(S.indptr)[rows]
    sub_indptr = np.concatenate([[0], np.cumsum(deg)]).astype(np.int64)
    eids = np.concatenate([np.arange(S.indptr[r], S.indptr[r + 1]) for r in rows]).astype(np.int64)
    uniq, local = np.unique(S.indices[eids], return_inverse=True)
    import torch
    take = torch.from_numpy(uniq).cuda().long()
    z = S.z[take, :f].cpu().numpy()
    if kind == "gat":
        el = S.el[h][torch.from_numpy(rows).cuda().long()].cpu().numpy()
        er = S.er[h][take].cpu().numpy()
        r = _gat_from_z(sub_indptr, local, z, el, er)
        return r["Y"], O.gat_rowscale(sub_indptr, local, z.astype(np.float64), r["alpha"])
    w = S.w[torch.from_numpy(eids).cuda().long()].cpu().numpy().astype(np.float64) if h else None
    return O.spmm(sub_indptr, local, w, z), O.spmm(sub_indptr, local, None if w is None else np.abs(w), np.abs(z))


@pytest.mark.parametrize("kind,f,h", STATIC_WIDE, ids=[f"{k}-f{f}-h{h}" for k, f, h in STATIC_WIDE])
def test_static_striding_through_exchange_in_every_window(static_world2, monkeypatch, kind, f, h):
    """World 2 on a low-degree graph with enough items for static striding, at widths that need a second feature
    window: in windows past the first the copy CTAs of window 0 do not exist, so the static cursor must stride over
    the whole grid there.  The static step must equal a dynamic step on the same data bit for bit, hold every slot, and
    match the oracle on a sample of rows."""
    import torch
    from gta_graph_tensor_acclelrator_for_general_gnn_b200 import kernels
    S = static_world2
    z = S.z[:, :f]

    def produce(p, ex):
        b0, b1 = p.row_begin, p.row_end
        if kind == "gat":
            zt, ert, gate = ex.gather_pair(z[b0:b1], S.er[h][b0:b1])
            return (zt, ert), gate
        table, gate = ex.gather_one(z[b0:b1])
        return (table,), gate

    def consume(p, tables, gate):
        if kind == "gat":
            el = S.el[h][p.row_begin:p.row_end].clone()          # the kernel takes el 16-byte aligned
            return kernels.gat_aggregate(p.local, el, tables[1], tables[0], exchange=gate)
        e0, e1 = int(S.indptr[p.row_begin]), int(S.indptr[p.row_end])
        return kernels.aggregate(p.local, tables[0], p.permute_edges(S.w[e0:e1]) if h else None, exchange=gate)

    wants = (z, S.er[h]) if kind == "gat" else (z,)
    monkeypatch.setattr(kernels, "STATIC_MIN_ITEMS", 1 << 62)          # dynamic item fetch
    dynamic = run_step(S.parts, S.exs, produce, consume)
    assert_slots_hold(S.parts, dynamic, wants, f"{kind} f={f} dynamic")
    monkeypatch.setattr(kernels, "STATIC_MIN_ITEMS", 0)
    monkeypatch.setattr(kernels, "STATIC_ITEM_EDGES", 1 << 30)
    static = run_step(S.parts, S.exs, produce, consume)
    assert_slots_hold(S.parts, static, wants, f"{kind} f={f} static")
    for p, (a, _, _), (b, _, _) in zip(S.parts, dynamic, static):
        assert a.equal(b), f"{kind} f={f}: rank {p.rank}'s static step differs from the dynamic one"
    out = _cat(static)
    rows = np.sort(np.random.default_rng(f).choice(S.n, 3000, replace=False))
    want, scale = _sample_oracle(S, kind, f, h, rows)
    got = out[torch.from_numpy(rows).cuda()].cpu().numpy()
    assert_close_rowscale(got, want, scale, what=f"{kind} f={f} static striding, sampled rows")
