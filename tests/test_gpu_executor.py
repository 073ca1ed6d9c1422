"""execute(): ISA programs emitted by the unmodified reference (tests/golden/isa) run on the
GPU and are compared with the op-by-op CPU oracle on the same synthetic graph."""
import json
import os

import numpy as np
import pytest
import yaml

from conftest import assert_close_rowscale
from oracle import gta_oracle as O
from gta_graph_tensor_acclelrator_for_general_gnn_b200 import synthetic
from test_gpu_kernels import _gat_from_z

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
with open(os.path.join(GOLDEN, "manifest.json")) as _f:
    MANIFEST = json.load(_f)
PROGRAMS = [p for p in MANIFEST["programs"]]


def _load(rel):
    with open(os.path.join(GOLDEN, rel)) as f:
        return yaml.safe_load(f)


def _small_shape(dataset):
    # programs generated for Flickr/Reddit shapes are exercised on a shrunken graph: the
    # executor ignores Tile_Times (an ASIC buffer decision), so only the op sizes change
    n, e, f = synthetic.SHAPES[dataset]
    if dataset == "cora":
        return n, e, f
    return 4000, 60000, f


def _inputs(op_info, n, e, seed=0):
    """Random tensors for every external input / weight of an op graph (fp32)."""
    return synthetic.opgraph_inputs(op_info, n, e, seed)


@pytest.fixture(scope="module")
def rt():
    import torch
    from gta_graph_tensor_acclelrator_for_general_gnn_b200 import executor, graph, isa, kernels

    class NS:
        pass
    ns = NS()
    ns.torch, ns.ex, ns.graph, ns.isa, ns.k = torch, executor, graph, isa, kernels
    return ns


_graph_cache = {}


def _graph(rt, dataset):
    if dataset not in _graph_cache:
        n, e, _ = _small_shape(dataset)
        g = synthetic.powerlaw_graph(n, e, seed=11, i0=20.0)
        indptr, indices, _ = O.csr_build(g.dst, g.src, n)
        dg = rt.graph.csr_from_coo(g.dst, g.src, n)
        _graph_cache[dataset] = (g, indptr, indices, dg)
    return _graph_cache[dataset]


@pytest.mark.parametrize("prog", PROGRAMS, ids=[p["file"].split("/")[-1][:-5] for p in PROGRAMS])
@pytest.mark.parametrize("fuse", [True, False], ids=["fused", "stores-honoured"])
def test_program_matches_oracle(rt, prog, fuse):
    op_info = _load(prog["opgraph"])
    records = _load(prog["file"])
    g, indptr, indices, dg = _graph(rt, prog["dataset"])
    n, e = g.num_nodes, g.num_edges
    node_inputs, weights, edge_inputs = _inputs(op_info, n, e)
    sem = O.NETWORK_SEMANTICS.get((prog["network"], prog["reorder"]), {})
    ref, ref_scale = O.run_opgraph(op_info, indptr, indices, node_inputs, weights, edge_inputs, semantics=sem,
                                   stabilize=True, return_scale=True)
    up = lambda v: [rt.torch.from_numpy(a).cuda() for a in v] if isinstance(v, list) else rt.torch.from_numpy(v).cuda()
    dev = lambda d: {k: up(v) for k, v in d.items()}
    out, log = rt.ex.execute(records, op_info, dg, dev(node_inputs), dev(weights), dev(edge_inputs),
                             network=prog["network"], is_reorder=prog["reorder"], fuse_across_blocks=fuse,
                             check_shapes=(prog["dataset"] == "cora"), return_log=True)
    finals = [p for p in range(len(op_info)) if not op_info[p]["OUTPUT"]["output_list"]]
    assert sorted(out) == finals
    for p in finals:
        y = out[p].cpu().numpy()
        y64 = ref[p]
        assert y.shape == y64.shape
        # the stated fp32 tolerance: 1e-5 |y64| + 1e-5 rowscale (first-order error scale of the op graph)
        assert_close_rowscale(y, y64, ref_scale[p], what=f"op {p}; kernels {log}")
    names = [k for k, _ in log]
    if prog["network"] == "GAT" and fuse:
        f_out, heads = op_info[0]["OUTPUT"]["size_per_feature"] // 4, op_info[1]["OUTPUT"]["size_per_feature"] // 4
        # the edge phase collapsed to one pass -- layer 3 of the reference's GAT (F = H = 16, one feature per head) too
        assert (f_out // heads) % 4 == 0 or f_out // heads in (1, 2)
        assert "gta_gat_aggregate_f32" in names, names
        assert not any(k.startswith("gta_edge_") for k in names), names
    if prog["network"] in ("GCN", "SGC", "GraphSAGE", "GIN"):
        assert any(k.startswith("gta_aggregate_f32") for k in names), names
        if fuse:        # E x Fin scatters stay virtual: no materialising copy, no generic edge kernel
            assert not any(k.startswith("gta_edge_") for k in names), names


def test_intermediate_outputs_on_request(rt):
    """Ask for GAT intermediates (S, alpha): they must be materialised and correct."""
    prog = next(p for p in PROGRAMS if p["network"] == "GAT" and p["dataset"] == "cora" and not p["reorder"]
                and len(p["op_array"]) == 3)
    op_info = _load(prog["opgraph"])
    g, indptr, indices, dg = _graph(rt, "cora")
    node_inputs, weights, edge_inputs = _inputs(op_info, g.num_nodes, g.num_edges)
    ref, ref_scale = O.run_opgraph(op_info, indptr, indices, node_inputs, weights, edge_inputs,
                                   semantics=O.NETWORK_SEMANTICS[("GAT", False)], stabilize=True, return_scale=True)
    dev = lambda d: {k: rt.torch.from_numpy(v).cuda() for k, v in d.items()}
    out = rt.ex.execute(_load(prog["file"]), op_info, dg, dev(node_inputs), dev(weights), dev(edge_inputs),
                        network="GAT", outputs=[8, 9, 13])
    for p in (8, 9, 13):
        assert_close_rowscale(out[p].cpu().numpy(), ref[p], ref_scale[p], what=f"op {p}")


def test_refuses_oversized_edge_tensor(rt):
    """GCN-original plan [[0],[1,2,3]] stores the E x Fin scatter (STORE_E FL=5732): with
    STORE_* honoured and a small budget the executor must refuse, not crash."""
    prog = next(p for p in PROGRAMS if p["file"].endswith("GCN-cora-layer1-original__0_1-2-3.yaml"))
    op_info = _load(prog["opgraph"])
    g, indptr, indices, dg = _graph(rt, "cora")
    node_inputs, weights, edge_inputs = _inputs(op_info, g.num_nodes, g.num_edges)
    dev = lambda d: {k: rt.torch.from_numpy(v).cuda() for k, v in d.items()}
    with pytest.raises(rt.ex.ExecutionError, match="max_edge_bytes"):
        rt.ex.execute(_load(prog["file"]), op_info, dg, dev(node_inputs), dev(weights), dev(edge_inputs),
                      network="GCN", fuse_across_blocks=False, max_edge_bytes=1 << 20)


def test_rejects_bad_programs(rt):
    prog = PROGRAMS[0]
    op_info = _load(prog["opgraph"])
    records = _load(prog["file"])
    g, _, _, dg = _graph(rt, "cora")
    bad = [[dict(records[0][0], TYPE="COMP_FOO")]]
    with pytest.raises(rt.isa.IsaError):
        rt.ex.execute(bad, op_info, dg, {}, {})
    legacy = [dict(op) for op in op_info]
    del legacy[0]["COMP_TYPE"]
    with pytest.raises(rt.isa.IsaError, match="COMP_TYPE"):
        rt.ex.execute(records, legacy, dg, {}, {})
    with pytest.raises(rt.ex.ExecutionError, match="generated for"):
        small = rt.graph.csr_from_coo(np.array([0, 1], np.int32), np.array([1, 0], np.int32), 2)
        rt.ex.execute(records, op_info, small, {}, {})


def test_chrome_timeline_export(rt, tmp_path):
    """GPU timeline in the simulator's chrome_timeline.json schema (simulator.py:360-382)."""
    from gta_graph_tensor_acclelrator_for_general_gnn_b200 import trace
    prog = next(p for p in PROGRAMS if p["file"].endswith("GCN-cora-layer1-trans__0_1-2-3.yaml"))
    op_info = _load(prog["opgraph"])
    g, _, _, dg = _graph(rt, "cora")
    node_inputs, weights, edge_inputs = _inputs(op_info, g.num_nodes, g.num_edges)
    dev = lambda d: {k: rt.torch.from_numpy(v).cuda() for k, v in d.items()}
    rt.k.EVENT_LOG = []
    try:
        _, log = rt.ex.execute(_load(prog["file"]), op_info, dg, dev(node_inputs), dev(weights), dev(edge_inputs),
                               network="GCN", is_reorder=True, return_log=True)
        path = trace.save_timeline(rt.k.EVENT_LOG, log, str(tmp_path))
    finally:
        rt.k.EVENT_LOG = None
    events = json.load(open(path))
    assert [e["name"] for e in events] == ["COMP_MM", "COMP_MUL_COMP_ADD"]
    assert [e["pid"] for e in events] == ["MM", "VEC_ALU"]
    assert all(e["ph"] == "X" and e["dur"] > 0 and set(e) == {"name", "cat", "ph", "ts", "dur", "pid", "tid"} for e in events)
    assert events[0]["ts"] == 0 and events[1]["ts"] >= events[0]["dur"] * 0.5


def test_host_pipeline_matches_direct_execution(rt):
    """pipeline.HostPipeline (copy-in / compute / copy-out streams, 2 staging buffers) returns exactly what
    execute() returns on resident inputs, for every batch of a sequence."""
    from gta_graph_tensor_acclelrator_for_general_gnn_b200 import pipeline
    torch = rt.torch
    prog = next(p for p in PROGRAMS if p["file"].endswith("GCN-cora-layer1-trans__0_1-2-3.yaml"))
    op_info = _load(prog["opgraph"])
    records = _load(prog["file"])
    g, _, _, dg = _graph(rt, "cora")
    n, fin = g.num_nodes, 1433
    node_inputs, weights, edge_inputs = _inputs(op_info, n, g.num_edges)
    dev = lambda d: {k: torch.from_numpy(v).cuda() for k, v in d.items()}
    w_d, e_d = dev(weights), dev(edge_inputs)

    def run(x_dev):
        return rt.ex.execute(records, op_info, dg, {0: x_dev}, w_d, e_d, network="GCN", is_reorder=True)[3]

    rng = np.random.default_rng(5)
    batches = [rng.standard_normal((n, fin), dtype=np.float32) for _ in range(5)]
    want = [run(rt.k.to_table(torch.from_numpy(b).cuda())).cpu() for b in batches]
    pipe = pipeline.HostPipeline(run, n, fin, "cuda", depth=2)
    xs, ys = [], []
    for b in batches:
        xp = pipeline.pinned_table(n, fin)
        xp.copy_(torch.from_numpy(b))
        xs.append(xp)
        ys.append(torch.empty((n, 128), dtype=torch.float32).pin_memory())
    for xp, yp in zip(xs, ys):
        pipe.submit(xp, yp)
    ms = pipe.finish()
    assert ms > 0
    for got, ref in zip(ys, want):
        assert torch.equal(got, ref)


# ---- the captured single-GPU step (executor.GraphedExecution) with different data at every replay -----------------------
GAT_PROGRAM = os.path.join("isa", "GAT-cora-layer1-original__0-1-2_4-5-6-7-8_3-9-10-11-12-13.yaml")
GCN_PROGRAM = os.path.join("isa", "GCN-cora-layer1-trans__0_1-2-3.yaml")
#: (program, op graph, network, reorder, final op, feature dtype); the bf16 GAT runs the 4-head op graph of the same
#: program (the bf16 single-pass kernel takes 1, 2 or 4 heads)
CAPTURED = {
    "gat-f32": (GAT_PROGRAM, "GAT-cora-layer1-original.yaml", "GAT", False, 13, "f32"),
    "gat-bf16": (GAT_PROGRAM, "GAT-cora-restamped-h4.yaml", "GAT", False, 13, "bf16"),
    "gcn-f32": (GCN_PROGRAM, "GCN-cora-layer1-trans.yaml", "GCN", True, 3, "f32"),
}
#: rows of the long chains in front of a graph of mean degree 100: 32, 10 and 4 items of 1024 edges, and 2
HUB_DEGREES = (32 * 1024 + 7, 10 * 1024, 4 * 1024 + 1, 1025)


@pytest.fixture(scope="module")
def big_graph(rt):
    """320 000 nodes of in-degree 100 behind four hub rows: a gathered table of 128 features is 164 MB in fp32 and
    82 MB in bf16, both above COL_BLOCK_THRESHOLD, and the mean degree allows two column blocks."""
    torch = rt.torch
    n, deg = 320_000, 100
    gen = torch.Generator(device="cuda").manual_seed(31)
    degs = torch.full((n,), deg, dtype=torch.int64, device="cuda")
    degs[:len(HUB_DEGREES)] = torch.tensor(HUB_DEGREES, device="cuda")
    dst = torch.repeat_interleave(torch.arange(n, dtype=torch.int32, device="cuda"), degs)
    src = torch.randint(0, n, (int(dst.shape[0]),), generator=gen, device="cuda", dtype=torch.int32)
    g = rt.graph.csr_from_coo(dst, src, n)
    indptr = g.indptr.cpu().numpy()
    rows = np.random.default_rng(31).choice(np.arange(len(HUB_DEGREES), n), 2000, replace=False)
    rows = np.sort(np.concatenate([np.arange(len(HUB_DEGREES)), rows]))
    eids = np.concatenate([np.arange(indptr[r], indptr[r + 1]) for r in rows])
    return g, n, rows, np.concatenate([[0], np.cumsum(np.diff(indptr)[rows])]).astype(np.int64), eids, \
        g.indices[torch.from_numpy(eids).cuda()].cpu().numpy().astype(np.int64)


def _stale_bound_overflows(sub_indptr, src, block_of_src, el_rows, er_src, er_stale_hi):
    """exp(e - b) is inf for some sampled edge when b = leaky(el + max er) takes the er maximum of each column block
    from another data set's statistics."""
    rows = O.row_ids(sub_indptr)
    e = O.leaky_relu(el_rows[rows].astype(np.float64) + er_src.astype(np.float64))
    b = O.leaky_relu(el_rows[rows].astype(np.float64) + er_stale_hi[block_of_src].astype(np.float64))
    with np.errstate(over="ignore"):
        return bool(np.any(np.isinf(np.exp((e - b).astype(np.float32)))))


@pytest.mark.parametrize("case", list(CAPTURED))
def test_captured_step_replays_changing_data(rt, big_graph, case):
    """execute() captured once into a CUDA graph, then d0, d1 = 30 d0, d2, d0 copied into the static input in place
    and replayed: every replay must match the fp64 oracle (on 2000 sampled rows and the hub rows of the longest chains),
    equal eager execute() on the same data bit for bit, and replay 4 must repeat replay 1.  d1 makes a softmax bound
    kept from d0's er statistics overflow exp, so a captured step that did not recompute them would show."""
    torch, k = rt.torch, rt.k
    prog, opname, network, reorder, final, dt = CAPTURED[case]
    g, n, rows, sub_indptr, eids, src = big_graph
    zdtype = torch.bfloat16 if dt == "bf16" else torch.float32
    f = 128
    assert g.schedule_for(k.pad_row(f, zdtype) * (2 if dt == "bf16" else 4)).num_blocks >= 2
    op_info, records = _load(os.path.join("opgraph", opname)), _load(prog)
    fin = op_info[0]["INPUT"]["size_per_feature"][0] // 4
    gen = torch.Generator(device="cuda").manual_seed(41)
    x0 = torch.randn((n, fin), generator=gen, device="cuda")
    data = [x0, x0 * 30.0, torch.randn((n, fin), generator=gen, device="cuda")]
    x_static = k.alloc_table(n, fin, "cuda")
    if network == "GAT":
        heads = op_info[1]["OUTPUT"]["size_per_feature"] // 4
        xs, w, al, ar = synthetic.gat_tensors(4096, fin, f, heads, seed=3)
        # er of d0 about N(0, 0.7): the bound path runs (a block's er range is far below 60), d1's er reaches about 30
        # times d0's maximum, which a bound kept from d0 cannot absorb, and |el + er| stays below 128, where half an fp32
        # ulp is 3.8e-6
        ar = (ar * (0.7 / float((xs @ w @ ar).std()))).astype(np.float32)
        weights = {0: torch.from_numpy(w).cuda(), 1: torch.from_numpy(al).cuda(), 2: torch.from_numpy(ar).cuda()}
        edge_inputs = None
    else:
        w = synthetic.glorot(np.random.default_rng(3), fin, f)
        weights = {0: torch.from_numpy(w).cuda()}
        deg = torch.diff(g.indptr).clamp(min=1).double()
        rows_of_edge = torch.repeat_interleave(torch.arange(n, device="cuda"), torch.diff(g.indptr))
        ew = (1.0 / torch.sqrt(deg[rows_of_edge] * deg[g.indices.long()])).float()
        edge_inputs = {2: ew[:, None].contiguous()}

    def step():
        return rt.ex.execute(records, op_info, g, {0: x_static}, weights, edge_inputs, network=network,
                             is_reorder=reorder, check_shapes=False, feature_dtype=zdtype)[final]

    x_static.copy_(data[0])
    graphed = rt.ex.GraphedExecution(step)
    sched = g.schedule_for(k.pad_row(f, zdtype) * (2 if dt == "bf16" else 4))
    block_of_src = src // sched.col_block
    take, local = np.unique(src, return_inverse=True)
    take_d, rows_d = torch.from_numpy(take).cuda(), torch.from_numpy(rows).cuda()
    replays, er_hi = [], {}
    for s, d in enumerate((0, 1, 2, 0)):
        what = f"{case} replay {s + 1} (d{d})"
        x_static.copy_(data[d])
        got = graphed.replay().clone()
        replays.append(got)
        eager = step()
        assert torch.equal(got, eager), f"{what}: differs from eager execute() on the same data"
        # fp64 oracle of the sampled rows, on the GEMM's own (fp32 or bf16-stored) Z and fp32 el / er
        if network == "GAT":
            z, el, er = k.gemm(k.to_table(data[d]), weights[0], weights[1], weights[2], z_dtype=zdtype)
            zs = z[take_d].float().cpu().numpy()
            el_rows, er_src = el[rows_d].cpu().numpy(), er[take_d].cpu().numpy()[local]
            r = _gat_from_z(sub_indptr, local, zs, el_rows, er[take_d].cpu().numpy())
            want = r["Y"]
            scale = O.gat_rowscale(sub_indptr, local, np.abs(zs).astype(np.float64), r["alpha"])
            er_hi[d] = torch.stack([er[sched.col_block * b: sched.col_block * (b + 1)].max(dim=0).values
                                    for b in range(sched.num_blocks)]).cpu().numpy()
            if d == 1:
                assert _stale_bound_overflows(sub_indptr, src, block_of_src, el_rows, er_src, er_hi[0]), \
                    f"{what}: a bound kept from d0's statistics would not overflow"
        else:
            zs = k.gemm(k.to_table(data[d]), weights[0])[take_d].cpu().numpy()
            wsub = edge_inputs[2][torch.from_numpy(eids).cuda(), 0].cpu().numpy().astype(np.float64)
            want = O.spmm(sub_indptr, local, wsub, zs)
            scale = O.spmm(sub_indptr, local, np.abs(wsub), np.abs(zs))
        assert_close_rowscale(got[rows_d].cpu().numpy(), want, scale, what=what)
    assert torch.equal(replays[0], replays[3]), f"{case}: replay 4 (d0 again) differs from replay 1"
