"""Every GEMM, GAT-logits, er-statistics and elementwise kernel instance, launched and held to an fp64 reference, and
an inventory that accounts for every kernel the built library holds.

The aggregation kernels have their own case table (test_gpu_instances.py).  Here GEMM_CASES names one call per row
together with the exact instances it must launch: gemm_tc_kernel<HMAX> (tcgen05 3xTF32; HMAX = 0, 4, 8, 16 by head
count) with its split_w_kernel pre-pass, or gemm_simt_kernel<BN> (FFMA) with attn_project_kernel when el / er are
asked for.  The tc rows run at N = 148 * 128 * 3 + 77, so every CTA of the persistent grid takes at least three tiles
(both TMEM accumulator buffers are reused) and the last tile is partial; F covers every multiple of 16 up to 256, so
the 4-, 3- and 2-stage rings all run.  test_every_library_kernel_is_claimed reads the kernel names of the built
library and fails on a kernel no table claims, on a claim for a kernel that does not exist, and on a table that no
longer covers the sweep it documents.
"""
import collections
import os
import re
import zlib

import numpy as np
import pytest

from conftest import assert_close_rowscale
from oracle import gta_oracle as O
from gta_graph_tensor_acclelrator_for_general_gnn_b200 import _cabi, synthetic
from test_gpu_instances import CASES, CRAFTED_DEGREES, kernel_instance, launched

TESTS = os.path.dirname(os.path.abspath(__file__))

# ---- kernel names: Itanium-mangled in the library, demangled in the profiler ----------------------------------------
_MANGLED_HEAD = re.compile(r"_ZN3gta(\d+)")
_MANGLED_ARGS = re.compile(r"I((?:Li\d+E)+)E")
_DEMANGLED = re.compile(r"\bgta::(\w+)(?:<([^<>]*)>)?\(")


def instance(name: str):
    """('gemm_tc_kernel', 4), ('split_w_kernel',), or an aggregation instance of test_gpu_instances, for a kernel
    name of namespace gta in either spelling; None for any other name."""
    inst = kernel_instance(name)
    if inst is not None:
        return inst
    m = _MANGLED_HEAD.search(name)
    if m:
        start = m.end() + int(m.group(1))
        args = _MANGLED_ARGS.match(name, start)
        return (name[m.end():start],) + (tuple(int(a) for a in re.findall(r"Li(\d+)E", args.group(1))) if args else ())
    m = _DEMANGLED.search(name)
    if m:
        args = m.group(2)
        return (m.group(1),) + (tuple(int(a.strip().replace("(int)", "")) for a in args.split(",")) if args else ())
    return None


def library_kernels(path: str = _cabi.LIB_PATH) -> set:
    """Every device kernel of namespace gta in the built library: its .text section names (host functions live in
    .text itself, and CUB's kernels are not in namespace gta)."""
    with open(path, "rb") as fh:
        return {instance(m.decode()) for m in re.findall(rb"\.text\.(_ZN3gta\w+)", fh.read())}


def test_dense_kernel_names_parse_in_every_spelling():
    assert instance("_ZN3gta14gemm_tc_kernelILi16EEEv14CUtensorMap_stS1_S1_NS_8TcParamsE") == ("gemm_tc_kernel", 16)
    assert instance("void gta::gemm_tc_kernel<(int)4>(CUtensorMap_st, CUtensorMap_st, CUtensorMap_st, gta::TcParams)") \
        == ("gemm_tc_kernel", 4)
    assert instance("void gta::gemm_simt_kernel<128>(float const*, long, float const*, long, float*, long, long, int, "
                    "int, int)") == ("gemm_simt_kernel", 128)
    assert instance("_ZN3gta14split_w_kernelEPKfliiiPfS2_") == ("split_w_kernel",)
    assert instance("gta::er_stats_kernel(float const*, long, long, long, int, unsigned int*)") == ("er_stats_kernel",)
    assert instance("_ZN3gta18edge_binary_kernelEPKlPKilliPKfiilS5_iilPfil") == ("edge_binary_kernel",)
    assert instance("void gta::aggregate_kernel<gta::Bf16x4, 2, 32, 1, true>(gta::WorkList, gta::Exchange)") == \
        ("aggregate_kernel", "Bf16x4", 2, 32, 1, True)
    assert instance("void at::native::vectorized_elementwise_kernel<4, at::native::FillFunctor<float>>(int, ...)") is None


# ---- the GEMM case table ------------------------------------------------------------------------------------------
# mode: gta_gemm_set_mode for the call ('auto' picks tc when eligible);  heads > 0 with attn 'lr' / 'l' / 'r' asks for
# el and er / el only / er only, with block-diagonal or dense Al / Ar (aw);  xl: X in a padded table whose pad columns
# hold NaN ('table'), contiguous with no pad ('k7'), or one column into a padded table ('offset', not 16-byte aligned);
# zl: Z in a table with sentinel pad columns and a sentinel row past N ('pad'), or Z and er as views of one
# [N, F | H | pad] table as the multi-GPU exchange lays them out ('dist');  z: 'bf16' rounds Z in the epilogue.
Gemm = collections.namedtuple("Gemm", "mode n k f heads attn aw xl zl z", defaults=(0, "", "block", "table", "pad", "f32"))

SMS = 148
NT = SMS * 128 * 3 + 77          # every CTA takes >= 3 tiles; the last tile is partial
NW = SMS * 128 + 1               # one CTA takes a second, one-row tile
F_SWEEP = tuple(range(16, 257, 16))
K_SWEEP = (1, 4, 31, 32, 33, 64, 602, 1433)
N_EDGES = (1, 127, 128, 129, SMS * 128, NW)
SIMT_F = (1, 8, 16, 17, 32, 33, 64, 65, 128, 129, 200, 500)
ATTN_SIMT = tuple((f, h) for f in (24, 128, 200) for h in (1, 3, 17, 32))


def TC(hmax):
    return frozenset({("split_w_kernel",), ("gemm_tc_kernel", hmax)})


def SIMT(f, attn=False):
    bn = 128 if f > 64 else 64 if f > 32 else 32 if f > 16 else 16
    return frozenset({("gemm_simt_kernel", bn)} | ({("attn_project_kernel",)} if attn else set()))


GEMM_CASES = (
    [(Gemm("tc", NT, 602, f), TC(0)) for f in F_SWEEP]
    + [(Gemm("tc", NW, k, 128), TC(0)) for k in K_SWEEP]
    + [(Gemm("tc", n, 33, 64), TC(0)) for n in N_EDGES]
    + [
        (Gemm("tc", NT, 602, 128, 1, "lr", "dense"), TC(4)),
        (Gemm("tc", 700, 602, 64, 2, "l"), TC(4)),
        (Gemm("tc", NW, 602, 48, 3, "r"), TC(4)),
        (Gemm("tc", NT, 602, 128, 4, "lr", zl="dist"), TC(4)),
        (Gemm("tc", 3000, 1433, 256, 4, "lr", "dense"), TC(4)),
        (Gemm("tc", NT, 602, 80, 5, "lr", zl="dist"), TC(8)),
        (Gemm("tc", 5000, 602, 128, 8, "l", "dense"), TC(8)),
        (Gemm("tc", NW, 602, 256, 8, "r"), TC(8)),
        (Gemm("tc", NT, 602, 144, 9, "lr", zl="dist"), TC(16)),
        (Gemm("tc", 3000, 602, 192, 12, "r", "dense"), TC(16)),
        (Gemm("tc", NT, 602, 176, 16, "lr", zl="dist"), TC(16)),          # 2 stages beside 22 KB of Al | Ar
        (Gemm("tc", 1000, 602, 256, 16, "l", "dense"), TC(16)),
        (Gemm("tc", NW, 602, 128, 16, "lr", "dense", zl="dist"), TC(16)),
    ]
    + [(Gemm("tc", NT, 602, f, 4, "lr", z="bf16"), TC(4)) for f in F_SWEEP]
    + [(Gemm("simt", 5000, 602, f), SIMT(f)) for f in SIMT_F]
    + [
        (Gemm("simt", 3000, 7, 65, xl="k7"), SIMT(65)),
        (Gemm("simt", 3000, 602, 33, xl="offset"), SIMT(33)),
        (Gemm("auto", 3000, 602, 128, xl="offset"), SIMT(128)),          # tc refuses an X that is not 16-byte aligned
        (Gemm("simt", 3000, 602, 200, 17, "lr", "dense", zl="dist"), SIMT(200, True)),
    ]
    + [(Gemm("simt", 3000, 602, f, h, "lr", "dense"), SIMT(f, True)) for f, h in ATTN_SIMT]
)


def _gemm_id(c):
    s = f"{c.mode}-n{c.n}-k{c.k}-f{c.f}"
    if c.heads:
        s += f"-h{c.heads}{c.attn}-{c.aw}"
    return s + "".join(f"-{v}" for v in (c.xl, c.zl, c.z) if v not in ("table", "pad", "f32"))


# ---- the other tables: kernels these tests launch, and kernels that existing tests run ------------------------------
TABLE_CLAIMS = {
    "test_gat_logits_match_fp64": {("gat_logits_kernel",)},
    "test_er_stats_on_a_strided_er": {("er_stats_kernel",)},
    "test_edge_binary_every_operand_kind": {("edge_binary_kernel",)},
    "test_edge_unary_every_op_and_kind": {("edge_unary_kernel",)},
    "test_node_ops_on_strided_tables": {("node_binary_kernel",), ("node_unary_kernel",)},
    "test_gather_peak_probe_runs": {("gather_peak_kernel",)},
}
ELSEWHERE = {
    ("pack_keys_kernel",): "test_gpu_kernels.py::test_csr_build_bit_exact",
    ("unpack_rows_kernel",): "test_gpu_kernels.py::test_csr_build_bit_exact",
    ("sched_count_kernel",): "test_gpu_kernels.py::test_schedule_covers_every_edge_once",
    ("sched_fill_kernel",): "test_gpu_kernels.py::test_schedule_covers_every_edge_once",
    ("tile_nnz_kernel",): "test_gpu_kernels.py::test_tile_nnz_against_reference_tables",
    ("max_i32_kernel",): "test_gpu_kernels.py::test_tile_nnz_against_reference_tables",
    ("partition_kernel",): "test_gpu_kernels.py::test_partition_and_reorder_bit_exact",
    ("degree_keys_kernel",): "test_gpu_kernels.py::test_partition_and_reorder_bit_exact",
    ("low_word_kernel",): "test_gpu_kernels.py::test_partition_and_reorder_bit_exact",
    ("remap_sources_kernel",): "test_gpu_dist.py::test_allgather_layout_equals_single_gpu",
    ("exchange_publish_kernel",): "test_gpu_exchange.py::test_instance_through_exchange_step_by_step",
    # the first aggregation call of a process reads the L2 eviction policy through it
    ("cache_policy_kernel",): "test_gpu_instances.py::test_instance_matches_fp64_oracle",
}


def _coverage_gaps():
    """What the GEMM table promises to cover (module docstring and the issue of each row), and what it misses."""
    gaps = []

    def need(what, have, want):
        missing = set(want) - set(have)
        if missing:
            gaps.append(f"{what}: missing {sorted(missing)}")
    plain = {(c.n, c.k, c.f) for c, _ in GEMM_CASES if c.mode == "tc" and not c.heads}
    need("tc F sweep", plain, [(NT, 602, f) for f in F_SWEEP])
    need("tc K sweep", plain, [(NW, k, 128) for k in K_SWEEP])
    need("tc N edges", plain, [(n, 33, 64) for n in N_EDGES])
    for hm, heads in ((4, (1, 2, 3, 4)), (8, (5, 8)), (16, (9, 12, 16))):
        rows = [c for c, inst in GEMM_CASES if ("gemm_tc_kernel", hm) in inst and c.z == "f32"]
        need(f"tc<{hm}> heads", {c.heads for c in rows}, heads)
        need(f"tc<{hm}> projections", {c.attn for c in rows}, ("lr", "l", "r"))
        need(f"tc<{hm}> Al/Ar forms", {c.aw for c in rows}, ("block", "dense"))
        need(f"tc<{hm}> multi-tile N", {c.n > SMS * 128 for c in rows}, (True,))
        need(f"tc<{hm}> exchange layout", {c.zl for c in rows}, ("dist",))
    attn = [c for c, _ in GEMM_CASES if c.mode == "tc" and c.heads and c.z == "f32"]
    need("tc attention at K = 1433", {c.k for c in attn}, (1433,))
    need("tc 16 heads at F >= 176, multi-tile", {c.heads for c in attn if c.f >= 176 and c.n > SMS * 128}, (16,))
    need("tc 16 heads at F >= 176, one tile per CTA", {c.heads for c in attn if c.f >= 176 and c.n <= SMS * 128}, (16,))
    need("tc 16 heads, dense Al/Ar in the exchange layout", {(c.heads, c.aw, c.zl) for c in attn}, [(16, "dense", "dist")])
    need("bf16 Z F sweep", {(c.n, c.f) for c, _ in GEMM_CASES if c.z == "bf16"}, [(NT, f) for f in F_SWEEP])
    simt = {(c.mode, c.n, c.k, c.f, c.heads, c.xl, c.zl) for c, _ in GEMM_CASES if c.mode != "tc"}
    need("simt F", simt, [("simt", 5000, 602, f, 0, "table", "pad") for f in SIMT_F])
    need("simt unaligned X", simt, [("simt", 3000, 7, 65, 0, "k7", "pad"), ("simt", 3000, 602, 33, 0, "offset", "pad"),
                                    ("auto", 3000, 602, 128, 0, "offset", "pad")])
    need("attn_project", simt, [("simt", 3000, 602, f, h, "table", "pad") for f, h in ATTN_SIMT] +
         [("simt", 3000, 602, 200, 17, "table", "dist")])
    return gaps


def test_every_library_kernel_is_claimed():
    """Every kernel of the built library is run by a case row here or in test_gpu_instances, or by the named existing
    test; a kernel without a claim, a claim for a kernel that does not exist, or a table that lost part of its sweep
    fails."""
    if not os.path.exists(_cabi.LIB_PATH):
        pytest.skip("the CUDA library has not been built")
    lib = library_kernels()
    claims = {inst for _, inst in CASES} | {k for _, insts in GEMM_CASES for k in insts} | set(ELSEWHERE)
    claims |= {k for insts in TABLE_CLAIMS.values() for k in insts}
    assert None not in lib, "a kernel name of the library does not parse"
    assert lib == claims, (f"{len(lib)} kernels; unclaimed: {sorted(lib - claims, key=repr)}; "
                           f"claimed but not in the library: {sorted(claims - lib, key=repr)}")
    with open(__file__) as fh:
        here = fh.read()
    for name in TABLE_CLAIMS:
        assert f"def {name}(" in here, f"TABLE_CLAIMS names {name}, which is not a test of this file"
    for kernel, where in ELSEWHERE.items():
        fname, test = where.split("::")
        with open(os.path.join(TESTS, fname)) as fh:
            assert f"def {test}(" in fh.read(), f"{kernel} is claimed by {where}, which does not exist"
    gaps = _coverage_gaps()
    assert not gaps, "; ".join(gaps)


# ---- device fixtures -----------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def D():
    import types

    import torch
    from gta_graph_tensor_acclelrator_for_general_gnn_b200 import graph, kernels
    _cabi.load()
    k = len(CRAFTED_DEGREES)
    graphs = {}
    for name, (n0, e0) in {"logits": (3000, 90000), "elementwise": (1200, 10000)}.items():
        g = synthetic.powerlaw_graph(n0, e0, seed=2, i0=3.0, name="skew")
        n = g.num_nodes + k
        rng = np.random.default_rng(23)
        dst = np.concatenate([np.full(d, r, np.int32) for r, d in enumerate(CRAFTED_DEGREES)] + [g.dst + k]).astype(np.int32)
        src = np.concatenate([rng.choice(n, d, replace=False).astype(np.int32) for d in CRAFTED_DEGREES] +
                             [g.src + k]).astype(np.int32)
        indptr, indices, _ = O.csr_build(dst, src, n)
        assert np.array_equal(np.diff(indptr)[:k], CRAFTED_DEGREES)
        graphs[name] = types.SimpleNamespace(n=n, e=len(indices), indptr=indptr, indices=indices, rows=O.row_ids(indptr),
                                             dg=graph.csr_from_coo(dst, src, n))
    return types.SimpleNamespace(torch=torch, k=kernels, **graphs)


def _dev(D, a):
    return D.torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _seed(*what):
    return zlib.crc32(repr(what).encode())


SENTINEL = -2.0 ** 100          # exact in fp32 and bf16


def _x(D, n, k, layout, kind, seed):
    """X [n, k] generated on the device from a seeded generator.  'table': pad columns hold NaN; 'k7': contiguous, no
    pad; 'offset': one column into a padded table of NaN.  kind 'normal', 'pos' (U(0,1)) or 'span' (N(0,1) rows scaled
    by 2^e, e in [-20, 20])."""
    torch = D.torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    if kind == "pos":
        v = torch.rand((n, k), generator=g, device="cuda")
    else:
        v = torch.randn((n, k), generator=g, device="cuda")
        if kind == "span":
            v *= torch.exp2(torch.randint(-20, 21, (n, 1), generator=g, device="cuda").float())
    if layout == "k7":
        return v
    buf = torch.full((max(n, 1), D.k.pad4(k + (layout == "offset"))), float("nan"), device="cuda")
    x = buf[:n, 1:1 + k] if layout == "offset" else buf[:n, :k]
    x.copy_(v)
    return x


def _checked_rows(n, seed):
    """Every row up to 4096; else the TMEM lane-quarter edges of every tile, the whole last tile and 2000 random rows."""
    if n <= 4096:
        return np.arange(n)
    tiles = (n + 127) // 128
    edges = (np.arange(tiles)[:, None] * 128 + np.array([0, 31, 32, 63, 64, 95, 96, 127])).ravel()
    rand = np.random.default_rng(seed).integers(0, n, 2000)
    rows = np.concatenate([edges, np.arange((tiles - 1) * 128, n), rand])
    return np.unique(rows[rows < n])


def _weights(c, seed, kind="normal"):
    rng = np.random.default_rng(seed)
    if kind == "pos":
        w = (rng.uniform(0, 1, (c.k, c.f)) / c.k).astype(np.float32)
    else:
        w = synthetic.glorot(rng, c.k, c.f)
    al = ar = None
    if c.heads:
        al, ar = (rng.uniform(-0.1, 0.1, (c.f, c.heads)).astype(np.float32) for _ in range(2))
        if c.aw == "block":          # head h sees only its own F / H slice
            mask = (np.arange(c.f)[:, None] * c.heads // c.f) == np.arange(c.heads)[None, :]
            al, ar = al * mask, ar * mask
        al, ar = (al if "l" in c.attn else None), (ar if "r" in c.attn else None)
    return w, al, ar


def _rowscale_check(D, got, rows_d, z64, zs, a, what):
    """got[rows] against fp64 Z (or Z.A when a is given), tolerance from |X|.|W| (.|A|)."""
    want, scale = (z64, zs) if a is None else (z64 @ a.astype(np.float64), zs @ np.abs(a).astype(np.float64))
    assert_close_rowscale(got.index_select(0, rows_d).float().cpu().numpy(), want, scale, what=what)


@pytest.fixture
def mode_restored(D):
    yield
    D.k.set_gemm_mode("auto")


@pytest.mark.gpu
@pytest.mark.parametrize("c,instances", GEMM_CASES, ids=[_gemm_id(c) for c, _ in GEMM_CASES])
def test_gemm_instance_matches_fp64(D, mode_restored, c, instances):
    torch, k = D.torch, D.k
    what = _gemm_id(c)
    seed = _seed(c)
    x = _x(D, c.n, c.k, c.xl, "normal", seed)
    w, al, ar = _weights(c, seed)
    wd, ald, ard = _dev(D, w), None if al is None else _dev(D, al), None if ar is None else _dev(D, ar)
    zdt = torch.bfloat16 if c.z == "bf16" else torch.float32
    h = c.heads
    if c.zl == "dist":          # Z and er in one [N, F | H | pad] fp32 table, as the exchange lays its slots out
        buf = torch.full((c.n + 1, k.pad4(c.f + h) + 4), SENTINEL, device="cuda")
        out, er_out = buf[:c.n, :c.f], buf[:c.n, c.f:c.f + h]
        written = [(slice(0, c.n), slice(0, c.f + (h if "r" in c.attn else 0)))]
    else:
        buf = torch.full((c.n + 1, k.pad_row(c.f, zdt) + (8 if c.z == "bf16" else 4)), SENTINEL, device="cuda", dtype=zdt)
        out, er_out = buf[:c.n, :c.f], None
        written = [(slice(0, c.n), slice(0, c.f))]
    a, b = min(131, c.n // 3), min(c.n, min(131, c.n // 3) + 1000)

    def call(xv, **kw):
        r = k.gemm(xv, wd, ald, ard, **kw)
        return r if isinstance(r, tuple) else (r, None, None)

    def run():
        k.set_gemm_mode(c.mode)
        full = call(x, out=out, er_out=er_out, z_dtype=zdt)
        again = call(x, z_dtype=zdt)
        part = call(x[a:b], z_dtype=zdt)
        f32 = call(x) if c.z == "bf16" else full
        return full, again, part, f32
    (full, again, part, f32), ran = launched(run, parse=instance)
    k.set_gemm_mode("auto")
    assert ran == instances, f"{what} launched {sorted(ran, key=repr)}, not {sorted(instances, key=repr)}"
    assert (full[1] is None) == (al is None) and (full[2] is None) == (ar is None)
    for t0, t1, t2, name in zip(full, again, part, "Z el er".split()):
        if t0 is None:
            continue
        assert torch.equal(t0, t1), f"{what}: {name} is not bitwise reproducible"
        assert torch.equal(t2, t0[a:b]), f"{what}: {name} of rows {a}:{b} differs from the same rows of the full call"
        assert bool(torch.isfinite(t0).all()), f"{what}: {name} is not finite (an X pad column was read?)"
    keep = torch.ones(buf.shape, dtype=torch.bool, device="cuda")
    for rs, cs in written:
        keep[rs, cs] = False
    assert bool((buf[keep] == SENTINEL).all()), f"{what}: a pad column or the row past N was written"
    if c.z == "bf16":
        assert torch.equal(full[0], f32[0].to(torch.bfloat16)), f"{what}: bf16 Z is not the rounded fp32 product"
        for t0, t32, name in zip(full[1:], f32[1:], ("el", "er")):
            assert torch.equal(t0, t32), f"{what}: {name} differs from the fp32 call's"
    rows = _checked_rows(c.n, seed)
    rows_d = torch.from_numpy(rows).cuda()
    xs = x.index_select(0, rows_d).cpu().numpy().astype(np.float64)
    z64 = xs @ w.astype(np.float64)
    zs = np.abs(xs) @ np.abs(w).astype(np.float64)
    _rowscale_check(D, f32[0], rows_d, z64, zs, None, what + " Z")
    if al is not None:
        _rowscale_check(D, f32[1], rows_d, z64, zs, al, what + " el")
    if ar is not None:
        _rowscale_check(D, f32[2], rows_d, z64, zs, ar, what + " er")


@pytest.mark.gpu
def test_gemm_refusals_come_before_any_launch(D, mode_restored):
    """Shapes outside the tc kernel's rules raise GtaUnsupported from host checks, with nothing launched; auto mode
    then runs the FFMA kernels and gets the right answer.  bf16 Z has no FFMA fallback, so there it always raises."""
    torch, k = D.torch, D.k
    lib = _cabi.load()
    n, kk = 700, 602
    x = _x(D, n, kk, "table", "normal", 11)
    xs = x.cpu().numpy().astype(np.float64)
    rng = np.random.default_rng(11)
    for f, heads in ((24, 0), (128, 17)):
        w = synthetic.glorot(rng, kk, f)
        al = ar = None
        if heads:
            al, ar = (rng.uniform(-0.1, 0.1, (f, heads)).astype(np.float32) for _ in range(2))
        args = (x, _dev(D, w)) + ((_dev(D, al), _dev(D, ar)) if heads else ())
        k.set_gemm_mode("tc")
        before = lib.gta_launch_count()
        with pytest.raises(_cabi.GtaUnsupported):
            k.gemm(*args)
        assert lib.gta_launch_count() == before, f"f={f} heads={heads}: a kernel launched before the refusal"
        k.set_gemm_mode("auto")
        got, ran = launched(lambda: k.gemm(*args), parse=instance)
        assert ran == SIMT(f, bool(heads))
        z, el, er = got if heads else (got, None, None)
        z64, zs = xs @ w.astype(np.float64), np.abs(xs) @ np.abs(w).astype(np.float64)
        assert_close_rowscale(z.cpu().numpy(), z64, zs, what=f"auto f={f} heads={heads} Z")
        if heads:
            for t, a, name in ((el, al, "el"), (er, ar, "er")):
                assert_close_rowscale(t.cpu().numpy(), z64 @ a.astype(np.float64), zs @ np.abs(a).astype(np.float64),
                                      what=f"auto f={f} heads={heads} {name}")
    for mode in ("auto", "tc"):
        k.set_gemm_mode(mode)
        for f in (24, 272):
            before = lib.gta_launch_count()
            with pytest.raises(_cabi.GtaUnsupported):
                k.gemm(x, _dev(D, synthetic.glorot(rng, kk, f)), z_dtype=torch.bfloat16)
            assert lib.gta_launch_count() == before, f"bf16 Z f={f}: a kernel launched before the refusal"


# Same-sign data is where an accumulator that truncates shows: the error then grows with K instead of cancelling.
PROBES = [("pos", 602), ("pos", 1433), ("pos", 4096), ("span", 602)]
#: the tcgen05 path's extra error per unit of K, relative to |X|.|W|: measured at about 1.2e-8 (4.7e-5 at K = 4096 on
#: same-sign data, NVIDIA B200 at 1000 W); include/gta_b200.h states the bound
TC_ACCUM_PER_K = 2.0 ** -26


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["tc", "simt"])
@pytest.mark.parametrize("kind,kk", PROBES, ids=[f"{a}-k{b}" for a, b in PROBES])
def test_gemm_accuracy_probe(D, mode_restored, mode, kind, kk):
    """X ~ U(0,1), W ~ U(0,1)/K (every term positive), or rows whose magnitudes span 2^-20 .. 2^20.  The FFMA path
    holds |z - z64| <= 1e-5 |z64| + 1e-5 |X|.|W|; the tcgen05 path that plus 2^-26 K |X|.|W|."""
    k = D.k
    c = Gemm(mode, 2048, kk, 128)
    seed = _seed(c, kind)
    x = _x(D, c.n, c.k, "table", kind, seed)
    w, _, _ = _weights(c, seed, kind if kind == "pos" else "normal")
    k.set_gemm_mode(mode)
    z = k.gemm(x, _dev(D, w)).cpu().numpy().astype(np.float64)
    k.set_gemm_mode("auto")
    xs = x.cpu().numpy().astype(np.float64)
    z64 = xs @ w.astype(np.float64)
    zs = np.abs(xs) @ np.abs(w).astype(np.float64)
    err = np.abs(z - z64)
    bound = 1e-5 * np.abs(z64) + (1e-5 + (TC_ACCUM_PER_K * kk if mode == "tc" else 0.0)) * zs
    print(f"accuracy probe {mode} {kind} K={kk}: max relative error {np.max(err / np.abs(z64)):.3e}, "
          f"{np.max(err / (1e-5 * np.abs(z64) + 1e-5 * zs)):.4f} of the fp32 tolerance, {np.max(err / bound):.4f} of "
          f"this path's bound")
    assert np.all(np.isfinite(z))
    assert np.max(err / bound) <= 1.0, f"{mode} {kind} K={kk}: {np.max(err / bound):.3f}x this path's bound"


# ---- GAT logits and er statistics -----------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("stabilize", [True, False])
@pytest.mark.parametrize("heads", [1, 2, 3, 4, 5, 8, 12, 16])
def test_gat_logits_match_fp64(D, heads, stabilize):
    """p = exp(leaky(el[i] + er[j]) - m[i]), with m the row max (stabilize) or 0, and the row sums, on rows that are
    empty, at the 32-lane edges and at 1023-1025 edges.  Stabilized, er spans about +-300 and all stays finite.
    The exponent argument is formed in fp32 as the kernel forms it; p may differ by expf's error and one rounding of
    that argument (leaky's product may be fused into the subtraction)."""
    torch, k, g = D.torch, D.k, D.logits
    rng = np.random.default_rng(_seed("logits", heads, stabilize))
    el = rng.standard_normal((g.n, heads), dtype=np.float32)
    er = rng.standard_normal((g.n, heads), dtype=np.float32) * np.float32(80 if stabilize else 1)
    eld, erd = _dev(D, el), _dev(D, er)
    (p, rowmax, rowsum), ran = launched(lambda: k.gat_logits(g.dg, eld, erd, stabilize=stabilize), parse=instance)
    assert ran == {("gat_logits_kernel",)}
    p2, m2, s2 = k.gat_logits(g.dg, eld, erd, stabilize=stabilize)
    assert torch.equal(p, p2) and torch.equal(rowmax, m2) and torch.equal(rowsum, s2), "not bitwise reproducible"
    p, rowmax, rowsum = (t.cpu().numpy() for t in (p, rowmax, rowsum))
    t = el[g.rows] + er[g.indices]                                  # fp32 sums, as the kernel forms them
    lr = np.where(t > 0, t, t * np.float32(k.LEAKY_SLOPE))
    mx = O.segment_max(lr.astype(np.float64), g.indptr)
    mx = np.where(np.isfinite(mx), mx, 0.0) if stabilize else np.zeros_like(mx)
    np.testing.assert_array_equal(rowmax, mx.astype(np.float32), err_msg="rowmax")
    arg = lr.astype(np.float64) - mx[g.rows]
    p64 = np.exp(arg)
    rel = 4 * 2.0 ** -23 + 2.0 ** -24 * (np.abs(lr) + np.abs(arg))          # expf, and one rounding of the argument
    assert np.all(np.isfinite(p)) and np.all(np.isfinite(rowsum))
    bad = np.abs(p - p64) > rel * p64 + 1e-43
    assert not bad.any(), f"p: {int(bad.sum())} entries off, e.g. edge {np.argwhere(bad)[0]}"
    s64 = O.segment_sum(p64, g.indptr)
    stol = O.segment_sum(rel * p64, g.indptr) + 1e-5 * s64
    bad = np.abs(rowsum - s64) > stol
    assert not bad.any(), f"rowsum: {int(bad.sum())} rows off, e.g. {np.argwhere(bad)[0]}"
    assert np.all(rowsum[np.diff(g.indptr) == 0] == 0)


def _decode(st):
    st = st.view(np.uint32)
    return np.where(st & 0x80000000, st & 0x7FFFFFFF, ~st).astype(np.uint32).view(np.float32)


@pytest.mark.gpu
@pytest.mark.parametrize("heads", [1, 2, 3, 4, 8, 16, 17, 32])
def test_er_stats_on_a_strided_er(D, heads):
    """er as the [F, F + H) columns of a wider table (lder > heads), whose neighbouring columns hold +-1e30: per column
    block, the decoded max er and max -er are exactly those of the block's rows.  Blocks of 701 do not divide N; blocks
    of N and N + 13 are one block.  A head count that is not a power of two has no statistics."""
    torch, k = D.torch, D.k
    n, f = D.logits.n, 20
    rng = np.random.default_rng(_seed("er_stats", heads))
    er = (rng.standard_normal((n, heads)) * 50).astype(np.float32)
    er.flat[::97] = -0.0
    er.flat[5::89] = 0.0
    tab = torch.full((n, k.pad4(f + heads) + 4), 1e30, device="cuda")
    tab[:, f + heads:] = -1e30
    erv = tab[:, f:f + heads]
    erv.copy_(_dev(D, er))
    if heads & (heads - 1):
        assert k.er_stats(erv) is None
        return
    for col_block in (0, 701, n, n + 13):
        st, ran = launched(lambda: k.er_stats(erv, col_block), parse=instance)
        assert ran == {("er_stats_kernel",)}
        dec = _decode(st.cpu().numpy())
        blocks = -(-n // col_block) if 0 < col_block < n else 1
        assert dec.shape == (blocks, 2, heads)
        for b in range(blocks):
            lo, hi = (b * col_block, min((b + 1) * col_block, n)) if blocks > 1 else (0, n)
            np.testing.assert_array_equal(dec[b, 0], er[lo:hi].max(axis=0), err_msg=f"col_block={col_block} block {b}")
            np.testing.assert_array_equal(-dec[b, 1], er[lo:hi].min(axis=0), err_msg=f"col_block={col_block} block {b}")


# ---- elementwise ----------------------------------------------------------------------------------------------------
KINDS = {"edge": _cabi.OPND_EDGE, "dst": _cabi.OPND_DST, "src": _cabi.OPND_SRC}
BINARY = {"add": _cabi.BIN_ADD, "mul": _cabi.BIN_MUL, "div": _cabi.BIN_DIV}
UNARY = {"exp_leaky": _cabi.UN_EXP_LEAKY_RELU, "elu": _cabi.UN_ELU, "relu": _cabi.UN_RELU, "copy": _cabi.UN_COPY}
EDGE_WIDTHS = [(w, w) for w in (1, 4, 31, 32, 33, 128)] + [(1, 128), (4, 128), (128, 4)]


def _binary64(op, a, b):
    """fp32 result of a correctly rounded fp32 op: the fp64 result rounded once (exact for + and *, and innocuous for
    / since 53 >= 2 * 24 + 2); division by +-0 is pinned to +0."""
    a, b = a.astype(np.float64), b.astype(np.float64)
    if op == "add":
        return (a + b).astype(np.float32)
    if op == "mul":
        return (a * b).astype(np.float32)
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.where(b != 0, a / np.where(b != 0, b, 1), 0.0).astype(np.float32)


def _operand(rng, op, rows, width, zeros):
    v = rng.standard_normal((rows, width), dtype=np.float32)
    if zeros:          # divisors of +0 and -0
        v.flat[::7] = 0.0
        v.flat[3::11] = -0.0
    return v


def _rows_of(g, kind, v):
    return {"edge": v, "dst": v[g.rows], "src": v[g.indices]}[kind]


@pytest.mark.gpu
@pytest.mark.parametrize("op", list(BINARY))
@pytest.mark.parametrize("ka", list(KINDS))
@pytest.mark.parametrize("kb", list(KINDS))
def test_edge_binary_every_operand_kind(D, op, ka, kb):
    """All 27 (op, kind_a, kind_b) combinations at widths on both sides of the flattened / per-column split (32), with
    head broadcast, compared bitwise with the correctly rounded fp32 result."""
    k, g = D.k, D.elementwise
    rng = np.random.default_rng(_seed("edge_binary", op, ka, kb))
    for wa, wb in EDGE_WIDTHS:
        wo = max(wa, wb)
        a = _operand(rng, op, g.e if ka == "edge" else g.n, wa, False)
        b = _operand(rng, op, g.e if kb == "edge" else g.n, wb, op == "div")
        out, ran = launched(lambda: k.edge_binary(g.dg, BINARY[op], _dev(D, a), KINDS[ka], _dev(D, b), KINDS[kb]),
                            parse=instance)
        assert ran == {("edge_binary_kernel",)}
        A = np.repeat(_rows_of(g, ka, a), wo // wa, axis=1)
        B = np.repeat(_rows_of(g, kb, b), wo // wb, axis=1)
        want = _binary64(op, A, B)
        got = out.cpu().numpy()
        assert got.shape == (g.e, wo)
        bad = got.view(np.uint32) != want.view(np.uint32)
        assert not bad.any(), f"{op} {ka}x{kb} wa={wa} wb={wb}: {int(bad.sum())} entries differ, e.g. {np.argwhere(bad)[0]}"


def _unary_check(op, got, a, slope, what):
    if op in ("relu", "copy"):
        want = np.maximum(a, np.float32(0)) if op == "relu" else a
        assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), what
        return
    if op == "exp_leaky":
        want = np.exp(np.where(a > 0, a, a * np.float32(slope)).astype(np.float64))
    else:
        want = np.where(a > 0, a.astype(np.float64), np.expm1(a.astype(np.float64)))
    ulp = np.spacing(np.abs(want).astype(np.float32)).astype(np.float64)
    bad = np.abs(got.astype(np.float64) - want) > 3 * ulp + 1e-45
    assert not bad.any(), f"{what}: {int(bad.sum())} entries beyond 3 ulp"


@pytest.mark.gpu
@pytest.mark.parametrize("op", list(UNARY))
@pytest.mark.parametrize("kind", list(KINDS))
def test_edge_unary_every_op_and_kind(D, op, kind):
    """Every edge-unary op on every operand kind; exp and ELU within 3 ulp of fp64 on the fp32 argument."""
    k, g = D.k, D.elementwise
    rng = np.random.default_rng(_seed("edge_unary", op, kind))
    for w in (1, 5, 33):
        a = rng.standard_normal((g.e if kind == "edge" else g.n, w), dtype=np.float32) * np.float32(4)
        out, ran = launched(lambda: k.edge_unary(g.dg, UNARY[op], _dev(D, a), KINDS[kind]), parse=instance)
        assert ran == {("edge_unary_kernel",)}
        _unary_check(op, out.cpu().numpy(), _rows_of(g, kind, a), k.LEAKY_SLOPE, f"{op} {kind} w={w}")


@pytest.mark.gpu
def test_node_ops_on_strided_tables(D):
    """Node binary (with head broadcast) and unary ops on tables whose pad columns hold NaN, which must not be read."""
    torch, k = D.torch, D.k
    n = D.elementwise.n
    rng = np.random.default_rng(_seed("node_ops"))

    def table(v):
        buf = torch.full((n, k.pad4(v.shape[1]) + 4), float("nan"), device="cuda")
        buf[:, :v.shape[1]].copy_(_dev(D, v))
        return buf[:, :v.shape[1]]
    ran_all = set()
    for op in BINARY:
        for wa, wb in ((5, 5), (1, 40), (40, 8), (128, 4), (33, 33)):
            wo = max(wa, wb)
            a = _operand(rng, op, n, wa, False)
            b = _operand(rng, op, n, wb, op == "div")
            out, ran = launched(lambda: k.node_binary(BINARY[op], table(a), table(b)), parse=instance)
            ran_all |= ran
            want = _binary64(op, np.repeat(a, wo // wa, axis=1), np.repeat(b, wo // wb, axis=1))
            got = out.cpu().numpy()
            assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), f"node {op} wa={wa} wb={wb}"
    for op in UNARY:
        for w in (5, 33):
            a = rng.standard_normal((n, w), dtype=np.float32) * np.float32(4)
            out, ran = launched(lambda: k.node_unary(UNARY[op], table(a)), parse=instance)
            ran_all |= ran
            _unary_check(op, out.cpu().numpy(), a, k.LEAKY_SLOPE, f"node {op} w={w}")
    assert ran_all == TABLE_CLAIMS["test_node_ops_on_strided_tables"]


@pytest.mark.gpu
def test_gather_peak_probe_runs(D):
    r, ran = launched(lambda: D.k.gather_peak(table_bytes=8 << 20, f=128, gathers_per_group=256, iters=1), parse=instance)
    assert ran - {("cache_policy_kernel",)} == {("gather_peak_kernel",)}          # the policy is read on first use
    assert r["gathers"] > 0 and r["gathers"] % 256 == 0 and r["ms"] > 0
