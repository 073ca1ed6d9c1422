"""Every compiled instance of the work-list aggregation kernels, launched and held to the fp64 oracle.

aggregate_kernel, gat_aggregate_kernel, gat_aggregate_llh_kernel and edge_sum_kernel are templates; which instance a
call runs depends on the storage type, the width, the weight kind, the head count and the terms.  CASES names one or
more calls per instance together with the instance each must launch.  The profiler reports the instance that really
ran, and test_case_table_is_the_library checks that the table's instances are exactly the ones the built library
holds: a new dispatch branch without a case here fails.

The graph is the power-law "skew" graph of test_gpu_kernels.py behind crafted rows whose degrees sit at every lane
count's batch edges (LANES - 1, LANES, LANES + 1) and at the item-chunk edges, and each case runs two work lists: short
items with long slot chains, and column blocks with chains that cross them.
"""
import os
import re
import zlib

import numpy as np
import pytest

from conftest import assert_close_rowscale
from oracle import gta_oracle as O
from gta_graph_tensor_acclelrator_for_general_gnn_b200 import _cabi, synthetic
from test_gpu_bf16 import _bf16_round
from test_gpu_kernels import _gat_from_z

FAMILY = ("aggregate_kernel", "gat_aggregate_kernel", "gat_aggregate_llh_kernel", "edge_sum_kernel")

# ---- instance names: Itanium-mangled in the library, demangled in the profiler ---------------------------------
_MANGLED = re.compile(rb"_ZN3gta(16aggregate_kernel|20gat_aggregate_kernel|24gat_aggregate_llh_kernel|15edge_sum_kernel)"
                      rb"I((?:NS_5F32x4E|NS_6Bf16x4E|NS_6Bf16x8E|Li\d+E|Lb[01]E)+)EEv")
_MANGLED_ARG = re.compile(rb"NS_\d(F32x4|Bf16x4|Bf16x8)E|Li(\d+)E|Lb([01])E")
_DEMANGLED = re.compile(r"\bgta::(" + "|".join(FAMILY) + r")<([^<>]*)>")


def _from_mangled(kernel: bytes, args: bytes) -> tuple:
    out = [kernel.lstrip(b"0123456789").decode()]
    for piece, i, b in _MANGLED_ARG.findall(args):
        out.append(piece.decode() if piece else (int(i) if i else b == b"1"))
    return tuple(out)


def _demangled_arg(a: str):
    a = a.strip()
    if a.startswith("gta::"):
        return a[len("gta::"):]
    if a in ("true", "(bool)1"):
        return True
    if a in ("false", "(bool)0"):
        return False
    return int(a[len("(int)"):] if a.startswith("(int)") else a)


def kernel_instance(name: str):
    """('aggregate_kernel', 'F32x4', 1, 32, 0, False) for a kernel name of the family (either spelling), else None."""
    m = _MANGLED.search(name.encode())
    if m:
        return _from_mangled(*m.groups())
    m = _DEMANGLED.search(name)
    if m:
        return (m.group(1),) + tuple(_demangled_arg(a) for a in m.group(2).split(","))
    return None


def library_instances(path: str = _cabi.LIB_PATH) -> set:
    """Every instance of the family that the built library holds, read from its symbol names."""
    with open(path, "rb") as fh:
        return {_from_mangled(*m) for m in _MANGLED.findall(fh.read())}


def launched(fn, parse=kernel_instance):
    """Run fn() under the profiler (CUDA activity only): returns (fn's result, set of instances that ran), an
    instance being whatever parse() makes of a kernel name (None: not one of the kernels looked for)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        result = fn()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events()]
    assert names, "the profiler recorded no kernels: which instance ran cannot be told"
    return result, {inst for inst in map(parse, names) if inst is not None}


# ---- the case table ------------------------------------------------------------------------------------------------
# calls:  ("aggregate", dtype, f, wh, div)  wh = 0: no weight, 1: scalar per edge, > 1: per head;  div: w / rowden
#         ("gat", dtype, f, heads)
#         ("edge_sum", f, terms, unary)      terms: e = edge [E, F], x = gathered sources, r = row term
def AGG(piece, v, lanes, wkind, div):
    return ("aggregate_kernel", piece, v, lanes, wkind, div)


def GAT(piece, lanes, heads):
    return ("gat_aggregate_kernel", piece, lanes, heads)


def LLH(lanes, heads_per_lane):
    return ("gat_aggregate_llh_kernel", lanes, heads_per_lane)


def ES(lanes, has_x, has_e):
    return ("edge_sum_kernel", lanes, has_x, has_e)


CASES = [
    # aggregate, fp32: lanes = pieces of 4 features up to 32; two pieces per lane above 128 features (not per head)
    (("aggregate", "f32", 16, 0, False), AGG("F32x4", 1, 4, 0, False)),
    (("aggregate", "f32", 16, 1, False), AGG("F32x4", 1, 4, 1, False)),
    (("aggregate", "f32", 16, 1, True), AGG("F32x4", 1, 4, 1, True)),
    (("aggregate", "f32", 16, 4, False), AGG("F32x4", 1, 4, 2, False)),
    (("aggregate", "f32", 16, 4, True), AGG("F32x4", 1, 4, 2, True)),
    (("aggregate", "f32", 32, 0, False), AGG("F32x4", 1, 8, 0, False)),
    (("aggregate", "f32", 24, 0, False), AGG("F32x4", 1, 8, 0, False)),
    (("aggregate", "f32", 32, 1, False), AGG("F32x4", 1, 8, 1, False)),
    (("aggregate", "f32", 30, 1, False), AGG("F32x4", 1, 8, 1, False)),          # padded to 32
    (("aggregate", "f32", 32, 1, True), AGG("F32x4", 1, 8, 1, True)),
    (("aggregate", "f32", 32, 4, False), AGG("F32x4", 1, 8, 2, False)),
    (("aggregate", "f32", 32, 4, True), AGG("F32x4", 1, 8, 2, True)),
    (("aggregate", "f32", 64, 0, False), AGG("F32x4", 1, 16, 0, False)),
    (("aggregate", "f32", 64, 1, False), AGG("F32x4", 1, 16, 1, False)),
    (("aggregate", "f32", 64, 1, True), AGG("F32x4", 1, 16, 1, True)),
    (("aggregate", "f32", 64, 2, False), AGG("F32x4", 1, 16, 2, False)),
    (("aggregate", "f32", 64, 4, True), AGG("F32x4", 1, 16, 2, True)),
    (("aggregate", "f32", 128, 0, False), AGG("F32x4", 1, 32, 0, False)),
    (("aggregate", "f32", 128, 1, False), AGG("F32x4", 1, 32, 1, False)),
    (("aggregate", "f32", 128, 1, True), AGG("F32x4", 1, 32, 1, True)),
    (("aggregate", "f32", 256, 4, False), AGG("F32x4", 1, 32, 2, False)),          # two 128-feature windows
    (("aggregate", "f32", 128, 2, False), AGG("F32x4", 1, 32, 2, False)),
    (("aggregate", "f32", 256, 4, True), AGG("F32x4", 1, 32, 2, True)),
    (("aggregate", "f32", 256, 0, False), AGG("F32x4", 2, 32, 0, False)),
    (("aggregate", "f32", 256, 1, False), AGG("F32x4", 2, 32, 1, False)),
    (("aggregate", "f32", 500, 1, False), AGG("F32x4", 2, 32, 1, False)),
    (("aggregate", "f32", 512, 1, True), AGG("F32x4", 2, 32, 1, True)),
    # aggregate, bf16 table: 8-byte pieces of 4 features, except rows wider than 128 in whole pieces of 8
    (("aggregate", "bf16", 16, 0, False), AGG("Bf16x4", 1, 4, 0, False)),
    (("aggregate", "bf16", 16, 1, False), AGG("Bf16x4", 1, 4, 1, False)),
    (("aggregate", "bf16", 16, 1, True), AGG("Bf16x4", 1, 4, 1, True)),
    (("aggregate", "bf16", 16, 4, False), AGG("Bf16x4", 1, 4, 2, False)),
    (("aggregate", "bf16", 16, 2, True), AGG("Bf16x4", 1, 4, 2, True)),
    (("aggregate", "bf16", 32, 0, False), AGG("Bf16x4", 1, 8, 0, False)),
    (("aggregate", "bf16", 30, 0, False), AGG("Bf16x4", 1, 8, 0, False)),          # padded to 32
    (("aggregate", "bf16", 32, 1, False), AGG("Bf16x4", 1, 8, 1, False)),
    (("aggregate", "bf16", 32, 1, True), AGG("Bf16x4", 1, 8, 1, True)),
    (("aggregate", "bf16", 32, 4, False), AGG("Bf16x4", 1, 8, 2, False)),
    (("aggregate", "bf16", 32, 8, True), AGG("Bf16x4", 1, 8, 2, True)),
    (("aggregate", "bf16", 64, 0, False), AGG("Bf16x4", 1, 16, 0, False)),
    (("aggregate", "bf16", 64, 1, False), AGG("Bf16x4", 1, 16, 1, False)),
    (("aggregate", "bf16", 64, 1, True), AGG("Bf16x4", 1, 16, 1, True)),
    (("aggregate", "bf16", 64, 4, False), AGG("Bf16x4", 1, 16, 2, False)),
    (("aggregate", "bf16", 64, 4, True), AGG("Bf16x4", 1, 16, 2, True)),
    (("aggregate", "bf16", 128, 0, False), AGG("Bf16x4", 1, 32, 0, False)),
    (("aggregate", "bf16", 128, 1, False), AGG("Bf16x4", 1, 32, 1, False)),
    (("aggregate", "bf16", 128, 1, True), AGG("Bf16x4", 1, 32, 1, True)),
    (("aggregate", "bf16", 128, 4, False), AGG("Bf16x4", 1, 32, 2, False)),
    (("aggregate", "bf16", 132, 3, False), AGG("Bf16x4", 1, 32, 2, False)),          # per-head width 44
    (("aggregate", "bf16", 128, 2, True), AGG("Bf16x4", 1, 32, 2, True)),
    (("aggregate", "bf16", 144, 4, True), AGG("Bf16x4", 1, 32, 2, True)),          # per-head width 36
    (("aggregate", "bf16", 132, 0, False), AGG("Bf16x4", 2, 32, 0, False)),
    (("aggregate", "bf16", 500, 0, False), AGG("Bf16x4", 2, 32, 0, False)),
    (("aggregate", "bf16", 260, 1, False), AGG("Bf16x4", 2, 32, 1, False)),
    (("aggregate", "bf16", 130, 1, False), AGG("Bf16x4", 2, 32, 1, False)),          # padded to 132
    (("aggregate", "bf16", 500, 1, True), AGG("Bf16x4", 2, 32, 1, True)),
    (("aggregate", "bf16", 256, 0, False), AGG("Bf16x8", 1, 32, 0, False)),
    (("aggregate", "bf16", 256, 1, False), AGG("Bf16x8", 1, 32, 1, False)),
    (("aggregate", "bf16", 256, 1, True), AGG("Bf16x8", 1, 32, 1, True)),
    (("aggregate", "bf16", 256, 4, False), AGG("Bf16x8", 1, 32, 2, False)),
    (("aggregate", "bf16", 256, 2, True), AGG("Bf16x8", 1, 32, 2, True)),
    (("aggregate", "bf16", 512, 0, False), AGG("Bf16x8", 2, 32, 0, False)),
    (("aggregate", "bf16", 512, 1, False), AGG("Bf16x8", 2, 32, 1, False)),
    (("aggregate", "bf16", 512, 1, True), AGG("Bf16x8", 2, 32, 1, True)),
    # staged GAT (H in 1, 2, 4, per-head width of whole pieces): windows of one 32-lane pass above that width
    (("gat", "f32", 16, 1), GAT("F32x4", 4, 1)),
    (("gat", "f32", 16, 2), GAT("F32x4", 4, 2)),
    (("gat", "f32", 16, 4), GAT("F32x4", 4, 4)),
    (("gat", "f32", 32, 1), GAT("F32x4", 8, 1)),
    (("gat", "f32", 32, 2), GAT("F32x4", 8, 2)),
    (("gat", "f32", 32, 4), GAT("F32x4", 8, 4)),
    (("gat", "f32", 64, 1), GAT("F32x4", 16, 1)),
    (("gat", "f32", 64, 2), GAT("F32x4", 16, 2)),
    (("gat", "f32", 64, 4), GAT("F32x4", 16, 4)),
    (("gat", "f32", 256, 1), GAT("F32x4", 32, 1)),
    (("gat", "f32", 512, 1), GAT("F32x4", 32, 1)),
    (("gat", "f32", 256, 2), GAT("F32x4", 32, 2)),
    (("gat", "f32", 512, 2), GAT("F32x4", 32, 2)),
    (("gat", "f32", 256, 4), GAT("F32x4", 32, 4)),
    (("gat", "f32", 512, 4), GAT("F32x4", 32, 4)),
    (("gat", "bf16", 16, 1), GAT("Bf16x4", 4, 1)),
    (("gat", "bf16", 16, 2), GAT("Bf16x4", 4, 2)),
    (("gat", "bf16", 16, 4), GAT("Bf16x4", 4, 4)),
    (("gat", "bf16", 32, 1), GAT("Bf16x4", 8, 1)),
    (("gat", "bf16", 32, 2), GAT("Bf16x4", 8, 2)),
    (("gat", "bf16", 32, 4), GAT("Bf16x4", 8, 4)),
    (("gat", "bf16", 64, 1), GAT("Bf16x4", 16, 1)),
    (("gat", "bf16", 64, 2), GAT("Bf16x4", 16, 2)),
    (("gat", "bf16", 64, 4), GAT("Bf16x4", 16, 4)),
    (("gat", "bf16", 128, 1), GAT("Bf16x4", 32, 1)),
    (("gat", "bf16", 132, 1), GAT("Bf16x4", 32, 1)),
    (("gat", "bf16", 136, 2), GAT("Bf16x4", 32, 2)),          # per-head width 68
    (("gat", "bf16", 128, 4), GAT("Bf16x4", 32, 4)),
    (("gat", "bf16", 144, 4), GAT("Bf16x4", 32, 4)),          # per-head width 36
    (("gat", "bf16", 256, 1), GAT("Bf16x8", 32, 1)),
    (("gat", "bf16", 256, 2), GAT("Bf16x8", 32, 2)),
    (("gat", "bf16", 256, 4), GAT("Bf16x8", 32, 4)),
    # lane-local-head GAT (fp32; any other head count): 1, 2 or 4 heads per lane for per-head widths 4k, 2, 1
    (("gat", "f32", 12, 3), LLH(4, 1)),
    (("gat", "f32", 8, 4), LLH(4, 2)),
    (("gat", "f32", 8, 8), LLH(4, 4)),
    (("gat", "f32", 32, 8), LLH(8, 1)),
    (("gat", "f32", 32, 16), LLH(8, 2)),
    (("gat", "f32", 32, 32), LLH(8, 4)),
    (("gat", "f32", 64, 16), LLH(16, 1)),
    (("gat", "f32", 48, 12), LLH(16, 1)),
    (("gat", "f32", 64, 32), LLH(16, 2)),
    (("gat", "f32", 48, 48), LLH(16, 4)),
    (("gat", "f32", 96, 6), LLH(32, 1)),
    (("gat", "f32", 256, 8), LLH(32, 1)),
    (("gat", "f32", 144, 12), LLH(32, 1)),          # head 10 straddles the two 128-feature windows
    (("gat", "f32", 128, 64), LLH(32, 2)),
    (("gat", "f32", 128, 128), LLH(32, 4)),
    # edge sum (fp32): lanes = pieces of 4 features up to 32; which of edge / x are present picks the instance
    (("edge_sum", 16, "exr", "relu"), ES(4, True, True)),
    (("edge_sum", 16, "xr", "elu"), ES(4, True, False)),
    (("edge_sum", 16, "er", "copy"), ES(4, False, True)),
    (("edge_sum", 16, "r", "relu"), ES(4, False, False)),
    (("edge_sum", 32, "ex", "elu"), ES(8, True, True)),
    (("edge_sum", 24, "exr", "relu"), ES(8, True, True)),
    (("edge_sum", 32, "x", "copy"), ES(8, True, False)),
    (("edge_sum", 30, "xr", "relu"), ES(8, True, False)),          # padded to 32
    (("edge_sum", 32, "e", "relu"), ES(8, False, True)),
    (("edge_sum", 32, "r", "elu"), ES(8, False, False)),
    (("edge_sum", 64, "exr", "elu"), ES(16, True, True)),
    (("edge_sum", 64, "xr", "relu"), ES(16, True, False)),
    (("edge_sum", 64, "er", "relu"), ES(16, False, True)),
    (("edge_sum", 64, "r", "copy"), ES(16, False, False)),
    (("edge_sum", 128, "exr", "relu"), ES(32, True, True)),
    (("edge_sum", 128, "x", "copy"), ES(32, True, False)),
    (("edge_sum", 128, "e", "elu"), ES(32, False, True)),
    (("edge_sum", 128, "r", "relu"), ES(32, False, False)),
]


def _case_id(call):
    if call[0] == "aggregate":
        _, dtype, f, wh, div = call
        return f"aggregate-{dtype}-f{f}-" + (f"w{wh}" if wh else "unweighted") + ("-div" if div else "")
    if call[0] == "gat":
        return "gat-{}-f{}-h{}".format(*call[1:])
    return "edge_sum-f{}-{}-{}".format(*call[1:])


def test_case_table_is_the_library():
    """The table reaches every instance the library compiles, and nothing else: a kernel instance without a case
    here is never run by the suite."""
    if not os.path.exists(_cabi.LIB_PATH):
        pytest.skip("the CUDA library has not been built")
    lib = library_instances()
    table = {inst for _, inst in CASES}
    assert len(lib) > 0
    assert table == lib, f"instances without a case: {sorted(lib - table)}; cases for no instance: {sorted(table - lib)}"


def test_instance_names_parse_in_every_spelling():
    want = ("aggregate_kernel", "Bf16x4", 2, 32, 1, True)
    assert kernel_instance("_ZN3gta16aggregate_kernelINS_6Bf16x4ELi2ELi32ELi1ELb1EEEvNS_8WorkListENS_8ExchangeE") == want
    assert kernel_instance("void gta::aggregate_kernel<gta::Bf16x4, 2, 32, 1, true>(gta::WorkList, gta::Exchange)") == want
    assert kernel_instance("void gta::aggregate_kernel<gta::Bf16x4, (int)2, (int)32, (int)1, (bool)1>(gta::WorkList)") == want
    assert kernel_instance("void gta::edge_sum_kernel<8, false, true>(gta::WorkList)") == ("edge_sum_kernel", 8, False, True)
    assert kernel_instance("void gta::gat_aggregate_kernel<gta::F32x4, 16, 2>(gta::WorkList)") == \
        ("gat_aggregate_kernel", "F32x4", 16, 2)
    assert kernel_instance("void gta::gat_aggregate_llh_kernel<(int)4, (int)1>(gta::WorkList)") == \
        ("gat_aggregate_llh_kernel", 4, 1)
    assert kernel_instance("void gta::er_stats_kernel(float const*, long, long, long, int, unsigned int*)") is None


# ---- the graph ---------------------------------------------------------------------------------------------------
#: degrees of the crafted rows in front of the skew graph: empty, single and short rows, one below / at / above a batch
#: of every lane count, and one below / at / above an item of 32 and 64 edges and of 1024
CRAFTED_DEGREES = sorted({0, 1, 3, 31, 32, 33, 63, 64, 65, 1023, 1024, 1025} |
                         {d for lanes in (4, 8, 16, 32) for d in (lanes - 1, lanes, lanes + 1)})
SCHEDULES = [(32, 0), (64, 700)]          # (chunk, col_block): long slot chains; column blocks with chains across them


def crafted_graph():
    g = synthetic.powerlaw_graph(3000, 90000, seed=2, i0=3.0, name="skew")
    k = len(CRAFTED_DEGREES)
    n = g.num_nodes + k
    rng = np.random.default_rng(23)
    dst = [np.full(d, r, np.int32) for r, d in enumerate(CRAFTED_DEGREES)] + [g.dst + k]
    src = [rng.choice(n, d, replace=False).astype(np.int32) for d in CRAFTED_DEGREES] + [g.src + k]
    return n, np.concatenate(dst).astype(np.int32), np.concatenate(src).astype(np.int32)


@pytest.fixture(scope="module")
def G():
    import types

    import torch
    from gta_graph_tensor_acclelrator_for_general_gnn_b200 import graph, kernels
    _cabi.load()
    n, dst, src = crafted_graph()
    indptr, indices, _ = O.csr_build(dst, src, n)
    assert np.array_equal(np.diff(indptr)[:len(CRAFTED_DEGREES)], CRAFTED_DEGREES)
    dg = graph.csr_from_coo(dst, src, n)
    return types.SimpleNamespace(torch=torch, k=kernels, n=n, e=len(indices), indptr=indptr, indices=indices,
                                 rows=O.row_ids(indptr), dg=dg, scheds=[dg.schedule(c, b) for c, b in SCHEDULES])


def _dev(G, a, dtype=None):
    t = G.torch.from_numpy(np.ascontiguousarray(a)).cuda()
    return t if dtype is None else t.to(dtype)


def _table(G, a, dtype="f32"):
    return G.k.to_table(_dev(G, a, G.torch.bfloat16 if dtype == "bf16" else None))


def _inputs(call, tag, shape):
    rng = np.random.default_rng(zlib.crc32(repr((call, tag)).encode()))
    return rng.standard_normal(shape, dtype=np.float32)


# ---- one runner per kernel family: launches under the profiler, then checks against fp64 -----------------------------
def _aggregate(G, call):
    _, dtype, f, wh, div = call
    x = _inputs(call, "x", (G.n, f))
    if dtype == "bf16":
        x = _bf16_round(x)          # the kernel sees exactly these values: fp32 tolerance
    w = rowden = weff = None
    if wh:
        w = np.random.default_rng(zlib.crc32(repr((call, "w")).encode())).uniform(0.1, 1.0, (G.e, wh)).astype(np.float32)
        weff = w.astype(np.float64)
        if div:          # a row's weight sum: 0 on an empty row, which must stay 0 rather than 0/0
            rowden = O.segment_sum(weff, G.indptr).astype(np.float32)
            weff = weff / rowden[G.rows]
    xd, wd, rd = _table(G, x, dtype), None if w is None else _dev(G, w), None if rowden is None else _dev(G, rowden)

    def run():
        return [(G.k.aggregate(G.dg, xd, wd, rd, sched=s), G.k.aggregate(G.dg, xd, wd, rd, sched=s)) for s in G.scheds]
    outs, ran = launched(run)
    want = O.spmm(G.indptr, G.indices, weff, x)
    scale = O.spmm(G.indptr, G.indices, None if weff is None else np.abs(weff), np.abs(x))
    for (chunk, col_block), (out, again) in zip(SCHEDULES, outs):
        what = f"{_case_id(call)} chunk={chunk} col_block={col_block}"
        assert out.shape == (G.n, f)
        assert G.torch.equal(out, again), f"{what}: not bitwise reproducible"
        assert_close_rowscale(out.cpu().numpy(), want, scale, what=what)
    return ran


def _gat(G, call):
    _, dtype, f, heads = call
    z = _inputs(call, "z", (G.n, f))
    if dtype == "bf16":
        z = _bf16_round(z)
    el = _inputs(call, "el", (G.n, heads))
    er = _inputs(call, "er", (G.n, heads))
    args = (G.dg, _dev(G, el), _dev(G, er), _table(G, z, dtype))

    def run():
        outs = []
        for s in G.scheds:
            bounded = G.k.gat_aggregate(*args, sched=s)
            outs.append((bounded, G.k.gat_aggregate(*args, sched=s), G.k.gat_aggregate(*args, sched=s, bounded=False),
                         G.k.gat_aggregate(*args, sched=s, want_stats=True)))
        return outs
    outs, ran = launched(run)
    r = _gat_from_z(G.indptr, G.indices, z, el, er)
    scale = O.gat_rowscale(G.indptr, G.indices, z.astype(np.float64), r["alpha"])
    has_er_stats = heads <= 32 and heads & (heads - 1) == 0
    for (chunk, col_block), (out_b, again, out_o, (out_s, rowmax, rowsum)) in zip(SCHEDULES, outs):
        what = f"{_case_id(call)} chunk={chunk} col_block={col_block}"
        assert G.torch.equal(out_b, again), f"{what}: bound path not bitwise reproducible"
        assert G.torch.equal(out_o, out_s), f"{what}: online path not bitwise reproducible"
        if not has_er_stats:          # no er statistics for this head count: the bound path IS the online path
            assert G.torch.equal(out_b, out_o), f"{what}: bounded and online differ without er statistics"
        assert_close_rowscale(out_b.cpu().numpy(), r["Y"], scale, what=what + " bounded")
        assert_close_rowscale(out_o.cpu().numpy(), r["Y"], scale, what=what + " online")
        np.testing.assert_allclose(rowmax.cpu().numpy(), r["rowmax"], rtol=1e-6, atol=1e-6, err_msg=what + " rowmax")
        np.testing.assert_allclose(rowsum.cpu().numpy(), r["S"], rtol=2e-5, err_msg=what + " rowsum")
    return ran


def _edge_sum(G, call):
    _, f, terms, unary = call
    edge = _inputs(call, "e", (G.e, f)) if "e" in terms else None
    x = _inputs(call, "x", (G.n, f)) if "x" in terms else None
    r = _inputs(call, "r", (G.n, f)) if "r" in terms else None
    v = np.zeros((G.e, f))
    sc = np.zeros((G.e, f))
    for t, sel in ((edge, slice(None)), (x, G.indices), (r, G.rows)):
        if t is not None:
            v = v + t[sel].astype(np.float64)
            sc = sc + np.abs(t[sel]).astype(np.float64)
    want = O.segment_sum({"relu": lambda a: np.maximum(a, 0), "elu": O.elu, "copy": lambda a: a}[unary](v), G.indptr)
    scale = O.segment_sum(sc, G.indptr)
    code = {"relu": _cabi.UN_RELU, "elu": _cabi.UN_ELU, "copy": _cabi.UN_COPY}[unary]
    tabs = [None if a is None else _table(G, a) for a in (edge, x, r)]

    def run():
        return [(G.k.aggregate_edge_sum(G.dg, *tabs, code, sched=s), G.k.aggregate_edge_sum(G.dg, *tabs, code, sched=s))
                for s in G.scheds]
    outs, ran = launched(run)
    for (chunk, col_block), (out, again) in zip(SCHEDULES, outs):
        what = f"{_case_id(call)} chunk={chunk} col_block={col_block}"
        assert out.shape == (G.n, f)
        assert G.torch.equal(out, again), f"{what}: not bitwise reproducible"
        assert_close_rowscale(out.cpu().numpy(), want, scale, what=what)
    return ran


@pytest.mark.gpu
@pytest.mark.parametrize("call,instance", CASES, ids=[_case_id(c) for c, _ in CASES])
def test_instance_matches_fp64_oracle(G, call, instance):
    ran = {"aggregate": _aggregate, "gat": _gat, "edge_sum": _edge_sum}[call[0]](G, call)
    assert ran == {instance}, f"{_case_id(call)} launched {sorted(ran)}, not {instance}"
