"""Destination-partitioned execution, all ranks emulated on ONE GPU.  No kernel here waits on a kernel that
has not been launched: every rank's producer + publish runs first, then every rank's aggregation -- whose copy
CTAs then find all peers ready.  (Real ranks, one GPU each: test_gpu_multiprocess.py.)"""
import numpy as np
import pytest

from conftest import assert_close_rowscale
from oracle import gta_oracle as O
from gta_graph_tensor_acclelrator_for_general_gnn_b200 import synthetic
from test_gpu_exchange import assert_slots_hold, emulated, release, run_step

pytestmark = pytest.mark.gpu


def _gat_case(n=3000, e=90000, fin=96, f=128, h=4):
    import torch
    from gta_graph_tensor_acclelrator_for_general_gnn_b200 import graph, kernels
    g = synthetic.powerlaw_graph(n, e, seed=2, i0=3.0)
    indptr, indices, _ = O.csr_build(g.dst, g.src, n)
    full = graph.csr_from_coo(g.dst, g.src, n)
    x, w, al, ar = synthetic.gat_tensors(n, fin, f, h, seed=1)
    dev = lambda a: torch.from_numpy(a).cuda()
    return indptr, indices, full, kernels.to_table(dev(x)), dev(w), dev(al), dev(ar), (x, w, al, ar)


@pytest.mark.parametrize("world", [2, 3, 8])
def test_allgather_layout_equals_single_gpu(world):
    """rotate=False (the NCCL all-gather layout, slot k = rank k): remapped ids stay ascending, so with the online
    softmax the rows every rank computes are the single-GPU rows bit for bit."""
    import torch
    from gta_graph_tensor_acclelrator_for_general_gnn_b200 import dist as gdist, kernels
    indptr, indices, full, xd, wd, ald, ard, _ = _gat_case()
    f, h = int(wd.shape[1]), int(ald.shape[1])
    z, el, er = kernels.gemm(xd, wd, ald, ard)
    want = kernels.gat_aggregate(full, el, er, z, bounded=False)
    want_bound = kernels.gat_aggregate(full, el, er, z)

    parts = [gdist.make_partition(full, r, world, rotate=False) for r in range(world)]
    bounds = parts[0].bounds
    assert bounds == [int(v) for v in O.partition_bounds(indptr, world)]
    stride = parts[0].stride
    assert stride % 8 == 0
    z_all = torch.zeros((world * stride, f), device="cuda")
    er_all = torch.zeros((world * stride, h), device="cuda")
    el_loc = []
    for p in parts:       # every rank's local GEMM, written into its slot of the gathered tables
        zl, ell, erl = kernels.gemm(xd[p.row_begin:p.row_end], wd, ald, ard)
        z_all[p.rank * stride: p.rank * stride + p.rows] = zl
        er_all[p.rank * stride: p.rank * stride + p.rows] = erl
        el_loc.append(ell)
        assert torch.equal(p.local.perm, torch.arange(p.local.num_edges, device="cuda"))      # order kept
    got = torch.cat([kernels.gat_aggregate(p.local, el_loc[p.rank], er_all, z_all, bounded=False) for p in parts])
    assert torch.equal(got, want)
    # bound path: the shift is taken from the gathered table (padding rows included): same values, maybe other bits
    got_b = torch.cat([kernels.gat_aggregate(p.local, el_loc[p.rank], er_all, z_all) for p in parts])
    assert torch.allclose(got_b, want_bound, rtol=1e-5, atol=1e-6)
    loads = [p.local.num_edges for p in parts]
    assert sum(loads) == full.num_edges and max(loads) - full.num_edges / world <= np.diff(indptr).max()


def test_er_beside_z_in_one_gathered_table():
    """The partitioned run ships [z | er] per source in ONE table; the GAT kernel reads er through its row
    stride.  Must equal the separate-table result bit for bit."""
    import torch
    from gta_graph_tensor_acclelrator_for_general_gnn_b200 import graph, kernels
    n, e, f, h = 3000, 90000, 128, 4
    g = synthetic.powerlaw_graph(n, e, seed=2, i0=3.0)
    full = graph.csr_from_coo(g.dst, g.src, n)
    rng = np.random.default_rng(0)
    z = torch.from_numpy(rng.standard_normal((n, f), dtype=np.float32)).cuda()
    el = torch.from_numpy(rng.standard_normal((n, h), dtype=np.float32)).cuda()
    er = torch.from_numpy(rng.standard_normal((n, h), dtype=np.float32)).cuda()
    want = kernels.gat_aggregate(full, el, er, kernels.to_table(z))
    table = torch.zeros((n, f + 4), device="cuda")
    table[:, :f] = z
    table[:, f:f + h] = er
    got = kernels.gat_aggregate(full, el, table[:, f:f + h], table[:, :f])
    assert torch.equal(got, want)


@pytest.mark.parametrize("world", [2, 4, 8])
@pytest.mark.parametrize("heads", [4, 8])
def test_fused_exchange_gat_emulated(world, heads):
    """The in-kernel exchange end to end on one GPU: per rank, GEMM straight into slot 0 of its table,
    gta_exchange_publish to every peer's signal block, then an aggregation launch whose first CTAs copy the
    peers' slots (here: other buffers of the same device) while the rest walk the work list behind the slot
    gates.  Three steps on X, another X, X again exercise both table parities with data that changes: every step must
    give the oracle's values for its own X, and step 3 the bits of step 1."""
    import torch
    from gta_graph_tensor_acclelrator_for_general_gnn_b200 import kernels
    indptr, indices, full, xd, wd, ald, ard, host = _gat_case(h=heads)
    x, w, al, ar = host
    f = int(wd.shape[1])
    x1 = np.random.default_rng(world * 10 + heads).standard_normal(x.shape, dtype=np.float32)
    data = {0: (x, xd), 1: (x1, torch.from_numpy(x1).cuda())}
    parts, exs = emulated(full, world, copy_ctas=8)
    outs = []
    for step, d in enumerate((0, 1, 0)):
        xs = data[d][1]

        def produce(p, ex):
            zv, erv = ex.local_views(f, heads, "cuda")
            z, el, er = kernels.gemm(xs[p.row_begin:p.row_end], wd, ald, ard, out=zv, er_out=erv)
            assert z.data_ptr() == zv.data_ptr() and er.data_ptr() == erv.data_ptr()
            zt, ert, gate = ex.gather_pair(z, er)
            assert gate.struct.step == step + 1 and gate.slot_rows == p.stride
            return (zt, ert), gate, el

        def consume(p, tables, gate, el):          # pull + reduce
            return kernels.gat_aggregate(p.local, el, tables[1], tables[0], exchange=gate)
        res = run_step(parts, exs, produce, consume)
        # after the launch every slot of every rank's table holds its owner's rows of this step (its owner's slot 0)
        own = [tables[0][:p.rows] for p, (_, tables, _) in zip(parts, res)]
        assert_slots_hold(parts, res, (torch.cat(own),), f"fused exchange world={world} H={heads} step={step + 1}")
        got = torch.cat([o for o, _, _ in res])
        outs.append(got)
        ref = O.gat_layer(indptr, indices, data[d][0], w, al, ar)
        zabs = np.abs(data[d][0]).astype(np.float64) @ np.abs(w).astype(np.float64)
        scale = O.segment_sum(O.head_broadcast(ref["alpha"], f) * zabs[indices], indptr)
        assert_close_rowscale(got.cpu().numpy(), ref["Y"], scale, what=f"fused exchange world={world} H={heads} step={step + 1}")
    assert torch.equal(outs[0], outs[2])
    release(exs)


@pytest.mark.parametrize("world", [2, 8])
def test_fused_exchange_gcn_emulated(world):
    """Same for the weighted aggregate (GCN): gather_one, edge weights permuted into the local edge order; Z changes
    from step to step."""
    import torch
    from gta_graph_tensor_acclelrator_for_general_gnn_b200 import graph, kernels
    n, e, f = 3000, 90000, 64
    g = synthetic.powerlaw_graph(n, e, seed=4, i0=3.0)
    indptr, indices, _ = O.csr_build(g.dst, g.src, n)
    full = graph.csr_from_coo(g.dst, g.src, n)
    rng = np.random.default_rng(2)
    zs = [rng.standard_normal((n, f), dtype=np.float32) for _ in range(2)]
    ew = synthetic.gcn_edge_norm(indptr, indices)
    ewd = torch.from_numpy(ew).cuda()
    parts, exs = emulated(full, world, copy_ctas=4)
    outs = []
    for step, d in enumerate((0, 1, 0)):
        zd = torch.from_numpy(zs[d]).cuda()

        def produce(p, ex):
            table, gate = ex.gather_one(zd[p.row_begin:p.row_end])
            return (table,), gate

        def consume(p, tables, gate):
            e0, e1 = int(indptr[p.row_begin]), int(indptr[p.row_end])
            return kernels.aggregate(p.local, tables[0], p.permute_edges(ewd[e0:e1]), exchange=gate)
        res = run_step(parts, exs, produce, consume)
        assert_slots_hold(parts, res, (zd,), f"fused GCN exchange world={world} step={step + 1}")
        got = torch.cat([o for o, _, _ in res])
        outs.append(got)
        want = O.spmm(indptr, indices, ew, zs[d])
        scale = O.spmm(indptr, indices, np.abs(ew), np.abs(zs[d]))
        assert_close_rowscale(got.cpu().numpy(), want, scale, what=f"fused GCN exchange world={world} step={step + 1}")
    assert torch.equal(outs[0], outs[2])
    release(exs)


def test_partition_from_coo_equals_make_partition():
    """Partition on build (degree histogram + one sort of the rank's own edges) gives the local graph
    make_partition cuts out of the replicated CSR."""
    import torch
    from gta_graph_tensor_acclelrator_for_general_gnn_b200 import dist as gdist, graph
    n, e, world = 3000, 90000, 4
    g = synthetic.powerlaw_graph(n, e, seed=6, i0=3.0)
    full = graph.csr_from_coo(g.dst, g.src, n)
    dst, src = torch.from_numpy(g.dst).cuda(), torch.from_numpy(g.src).cuda()
    for rank in range(world):
        for rotate in (False, True):
            a = gdist.make_partition(full, rank, world, rotate=rotate)
            b = gdist.partition_from_coo(dst, src, n, rank, world, rotate=rotate)
            assert a.bounds == b.bounds and a.stride == b.stride
            assert torch.equal(a.local.indptr, b.local.indptr) and torch.equal(a.local.indices, b.local.indices)


def test_split_launch_crosses_chains():
    """Column block 0 in one launch, the rest in a second (the chain flags are cleared once, before the first):
    same bits as the single launch."""
    import torch
    from gta_graph_tensor_acclelrator_for_general_gnn_b200 import graph, kernels
    n, e, f, h = 3000, 90000, 128, 4
    g = synthetic.powerlaw_graph(n, e, seed=2, i0=3.0)
    full = graph.csr_from_coo(g.dst, g.src, n)
    rng = np.random.default_rng(3)
    z, el, er = (torch.from_numpy(rng.standard_normal(s, dtype=np.float32)).cuda() for s in ((n, f), (n, h), (n, h)))
    sched = full.schedule(col_block=800)
    assert sched.num_blocks == 4
    a = kernels.gat_aggregate(full, el, er, z, sched=sched, block_events=[None] * 4)     # stats unknown: online softmax
    b = kernels.gat_aggregate(full, el, er, z, sched=sched, bounded=False)
    assert torch.equal(a, b)
    w = torch.rand(e, device="cuda")
    assert torch.equal(kernels.aggregate(full, z, w, sched=sched, block_events=[None] * 4),
                       kernels.aggregate(full, z, w, sched=sched))


def test_schedule_cut_points_equal_uniform_blocks():
    """gta_schedule_build_cuts with cut points at multiples of a block size is gta_schedule_build with that block
    size; uneven cuts (an exchange's slot groups) keep every edge exactly once, in order, inside its block."""
    import torch
    from gta_graph_tensor_acclelrator_for_general_gnn_b200 import dist as gdist, graph
    n, e = 3000, 90000
    g = synthetic.powerlaw_graph(n, e, seed=8, i0=3.0)
    full = graph.csr_from_coo(g.dst, g.src, n)
    a = full.schedule(col_block=800)
    b = full.schedule(col_cuts=(800, 1600, 2400))
    assert a.num_items == b.num_items and a.num_slots == b.num_slots and a.block_begin == b.block_begin
    assert torch.equal(a.items[:a.num_items], b.items[:b.num_items]) and torch.equal(a.row_slots, b.row_slots)
    cuts = (500, 2000)
    c = full.schedule(col_cuts=cuts)
    items = c.items[:c.num_items].cpu().numpy()
    indices = full.indices.cpu().numpy()
    assert items[:, 2].sum() == e and c.num_blocks == 3
    bounds = (0,) + cuts + (n,)
    for blk in range(3):
        for it in items[c.block_begin[blk]:c.block_begin[blk + 1]]:
            srcs = indices[it[1]:it[1] + it[2]]
            assert srcs.size == 0 or (srcs[0] >= bounds[blk] and srcs[-1] < bounds[blk + 1])
    assert gdist.slot_groups(8) == [[0], [1, 2, 3], [4, 5, 6, 7]] and gdist.slot_groups(2) == [[0], [1]]


@pytest.mark.parametrize("world", [2, 4])
def test_fused_exchange_bf16_tables_emulated(world):
    """bf16 storage mode across ranks: the IPC tables hold [Z bf16 | er fp32] rows (half the bytes of the pull), the GEMM
    rounds Z into slot 0, the bf16 gather kernel reads the pulled slots.  X changes from step to step.  Against the fp64
    oracle at the mode's tolerance, and against the single-GPU bf16 run at the fp32 tolerance (same stored values, other
    reduction order)."""
    import torch
    from gta_graph_tensor_acclelrator_for_general_gnn_b200 import kernels
    indptr, indices, full, xd, wd, ald, ard, host = _gat_case()
    x, w, al, ar = host
    f, heads = int(wd.shape[1]), int(ald.shape[1])
    x1 = np.random.default_rng(world).standard_normal(x.shape, dtype=np.float32)
    data = {0: (x, xd), 1: (x1, torch.from_numpy(x1).cuda())}
    parts, exs = emulated(full, world, copy_ctas=8)
    outs = []
    for step, d in enumerate((0, 1, 0)):
        xh, xs = data[d]
        ref = O.gat_layer(indptr, indices, xh, w, al, ar)
        zabs = np.abs(xh).astype(np.float64) @ np.abs(w).astype(np.float64)
        scale = O.segment_sum(O.head_broadcast(ref["alpha"], f) * zabs[indices], indptr)
        z1, el1, er1 = kernels.gemm(xs, wd, ald, ard, z_dtype=torch.bfloat16)
        single = kernels.gat_aggregate(full, el1, er1, z1).cpu().numpy()

        def produce(p, ex):
            zv, erv = ex.local_views(f, heads, "cuda", torch.bfloat16)
            assert zv.dtype == torch.bfloat16 and erv.dtype == torch.float32
            z, el, er = kernels.gemm(xs[p.row_begin:p.row_end], wd, ald, ard, out=zv, er_out=erv)
            zt, ert, gate = ex.gather_pair(z, er)
            assert gate.struct.row_bytes == 2 * f + 16 and zt.dtype == torch.bfloat16
            return (zt, ert), gate, el

        def consume(p, tables, gate, el):
            return kernels.gat_aggregate(p.local, el, tables[1], tables[0], exchange=gate)
        res = run_step(parts, exs, produce, consume)
        own = [tables[0][:p.rows] for p, (_, tables, _) in zip(parts, res)]
        assert_slots_hold(parts, res, (torch.cat(own),), f"bf16 exchange world={world} step={step + 1}")
        got_t = torch.cat([o for o, _, _ in res])
        outs.append(got_t)
        got = got_t.cpu().numpy()
        bound = 2e-2 * np.abs(ref["Y"]) + 1e-2 * scale + 1e-30
        assert np.all(np.isfinite(got)) and np.max(np.abs(got - ref["Y"]) / bound) <= 1.0
        assert_close_rowscale(got, single.astype(np.float64), scale, what=f"bf16 exchange world={world} step={step + 1}")
    assert torch.equal(outs[0], outs[2])
    release(exs)
