"""Parity of every CUDA entry point (through the C ABI) against the CPU oracle."""
import numpy as np
import pytest

from conftest import assert_close_rowscale
from oracle import gta_oracle as O
from gta_graph_tensor_acclelrator_for_general_gnn_b200 import synthetic

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def T():
    import torch
    from gta_graph_tensor_acclelrator_for_general_gnn_b200 import _cabi, graph, kernels
    _cabi.load()

    class NS:
        pass
    ns = NS()
    ns.torch, ns.cabi, ns.graph, ns.k = torch, _cabi, graph, kernels
    return ns


def _dev(T, a):
    return T.torch.from_numpy(np.ascontiguousarray(a)).cuda()


GRAPHS = [
    ("tiny", 64, 300, 1, 5.0),
    ("cora", 2708, 10556, 0, 100.0),
    ("skew", 3000, 90000, 2, 3.0),      # a few very long rows -> multi-item rows with chunk 32/1024
]


def _graph(name, n, e, seed, i0):
    return synthetic.powerlaw_graph(n, e, seed=seed, i0=i0, name=name)


@pytest.mark.parametrize("name,n,e,seed,i0", GRAPHS)
def test_csr_build_bit_exact(T, name, n, e, seed, i0):
    g = _graph(name, n, e, seed, i0)
    indptr, indices, perm = O.csr_build(g.dst, g.src, n)
    dg = T.graph.csr_from_coo(g.dst, g.src, n, want_perm=True)
    assert np.array_equal(dg.indptr.cpu().numpy(), indptr)
    assert np.array_equal(dg.indices.cpu().numpy(), indices)
    assert np.array_equal(dg.perm.cpu().numpy(), perm)


def test_damaged_edge_lists_are_refused_not_crashed_on(T):
    """A destination outside [0, N) or a negative id (ADVICE r1: unpack_rows_kernel used to write row pointers out of
    bounds for them) comes back as GTA_ERR_INVALID; duplicate edges make the tile tables refuse (the reference's
    tables count non-zeros of a dense adjacency)."""
    dst = np.array([0, 1, 2, 3], dtype=np.int32)
    src = np.array([1, 2, 3, 0], dtype=np.int32)
    for bad_dst, bad_src in (([0, 1, 2, 6], src), ([0, -1, 2, 3], src), (dst, [1, 2, -3, 0]), ([0, 1, 2, 2**31 - 1], src)):
        with pytest.raises(T.cabi.GtaError, match="outside"):
            T.graph.csr_from_coo(np.asarray(bad_dst, dtype=np.int32), np.asarray(bad_src, dtype=np.int32), 6)
    ok = T.graph.csr_from_coo(dst, src, 6)          # the library is still usable afterwards
    assert ok.num_edges == 4
    multi = T.graph.csr_from_coo(np.array([0, 0, 1], dtype=np.int32), np.array([2, 2, 0], dtype=np.int32), 3)
    with pytest.raises(ValueError, match="duplicate"):
        T.graph.calculate_sparsity(multi, 2)
    with pytest.raises(ValueError, match="duplicate"):
        T.graph.cal_min_sparsity(multi, 2)


def test_csr_build_duplicates_and_empty(T):
    # duplicate edges keep input order (stable); isolated nodes give empty rows
    dst = np.array([3, 1, 3, 3, 0, 1], dtype=np.int32)
    src = np.array([2, 0, 2, 1, 4, 0], dtype=np.int32)
    indptr, indices, perm = O.csr_build(dst, src, 6)
    dg = T.graph.csr_from_coo(dst, src, 6, want_perm=True)
    assert np.array_equal(dg.indptr.cpu().numpy(), indptr)
    assert np.array_equal(dg.indices.cpu().numpy(), indices)
    assert np.array_equal(dg.perm.cpu().numpy(), perm)
    empty = T.graph.csr_from_coo(np.zeros(0, np.int32), np.zeros(0, np.int32), 5)
    assert np.array_equal(empty.indptr.cpu().numpy(), np.zeros(6, np.int64))


def test_graph_without_rows(T):
    """The local graph of a rank whose edge-balanced range is empty: 0 nodes give indptr = [0] and a work list of 0
    items, and the calls of a step on it (GEMM over 0 rows, aggregations over 0 items, with the NULL data pointer of an
    empty edge-weight tensor) return empty outputs without a launch.  An edge into a 0-node graph is refused."""
    torch, k = T.torch, T.k
    g = T.graph.csr_from_coo(np.zeros(0, np.int32), np.zeros(0, np.int32), 0, want_perm=True)
    assert g.num_rows == 0 and g.num_edges == 0 and g.indptr.cpu().tolist() == [0]
    assert g.schedule().num_items == 0 and g.schedule(col_cuts=(8, 16)).num_items == 0
    with pytest.raises(T.cabi.GtaError, match="outside"):
        T.graph.csr_from_coo(np.zeros(1, np.int32), np.zeros(1, np.int32), 0)
    g.num_sources = 16
    lib = T.cabi.load()
    x = torch.zeros((0, 64), device="cuda")
    w = torch.randn(64, 32, device="cuda")
    al, ar = torch.randn(32, 4, device="cuda"), torch.randn(32, 4, device="cuda")
    table = k.alloc_table(16, 32, "cuda", zero=True)
    er_table = torch.zeros((16, 4), device="cuda")
    torch.cuda.synchronize()
    lib.gta_launch_count_reset()
    z, el, er = k.gemm(x, w, al, ar)
    assert z.shape == (0, 32) and el.shape == (0, 4) and er.shape == (0, 4)
    ew = torch.empty((0, 1), device="cuda")
    assert ew.data_ptr() == 0          # what a rank without edges hands the weighted aggregate
    assert k.aggregate(g, table, ew).shape == (0, 32)
    assert k.aggregate(g, table).shape == (0, 32)
    assert k.gat_aggregate(g, el, er_table, table).shape == (0, 32)
    out, rowmax, rowsum = k.gat_aggregate(g, el, er_table, table, want_stats=True)
    assert out.shape == (0, 32) and rowmax.shape == (0, 4) and rowsum.shape == (0, 4)
    assert int(lib.gta_launch_count()) == 0


def test_tile_nnz_against_reference_tables(T, golden_dir):
    import os
    for tag in ("g300", "g97"):
        z = np.load(os.path.join(golden_dir, "tiles", f"{tag}.npz"))
        n = int(z["num_nodes"])
        dg = T.graph.csr_from_coo(z["dst"], z["src"], n)
        for key in z.files:
            if not key.startswith("table_"):
                continue
            sr = int(key.split("_")[1])
            got = T.graph.calculate_sparsity(dg, sr).cpu().numpy()
            assert np.array_equal(got, z[key]), f"{tag} tile {sr}"
            assert T.graph.cal_min_sparsity(dg, sr) == int(z[key].max())
            # streamed in tiny batches must agree too
            assert T.graph.cal_min_sparsity(dg, sr, workspace_bytes=256 + 4 * n) == int(z[key].max())


@pytest.mark.parametrize("parts", [1, 2, 3, 8])
def test_partition_and_reorder_bit_exact(T, parts):
    g = _graph("skew", 3000, 90000, 2, 3.0)
    indptr, _, _ = O.csr_build(g.dst, g.src, g.num_nodes)
    dg = T.graph.csr_from_coo(g.dst, g.src, g.num_nodes)
    assert np.array_equal(T.graph.partition_bounds(dg, parts).cpu().numpy(), O.partition_bounds(indptr, parts))
    assert np.array_equal(T.graph.degree_reorder(dg).cpu().numpy(), O.degree_reorder(indptr))


@pytest.mark.parametrize("chunk", [32, 1024])
@pytest.mark.parametrize("col_block", [0, 700, 64])
def test_schedule_covers_every_edge_once(T, chunk, col_block):
    g = _graph("skew", 3000, 90000, 2, 3.0)
    indptr, indices, _ = O.csr_build(g.dst, g.src, g.num_nodes)
    dg = T.graph.csr_from_coo(g.dst, g.src, g.num_nodes)
    s = dg.schedule(chunk, col_block)
    items = s.items.cpu().numpy()[:s.num_items]
    row_slots = s.row_slots.cpu().numpy()
    n = g.num_nodes
    # expected item count: per (row, column block) segment, ceil(len / chunk); empty rows get one item
    blk = (indices // col_block) if col_block else np.zeros_like(indices)
    n_cb = int(-(-n // col_block)) if col_block else 1
    seg = np.bincount(O.row_ids(indptr) * n_cb + blk, minlength=n * n_cb).reshape(n, n_cb)
    per_row = (-(-seg // chunk)).sum(axis=1)
    per_row[per_row == 0] = 1
    assert s.num_items == int(per_row.sum())
    assert s.num_slots == int(per_row[per_row > 1].sum())
    assert np.array_equal(np.diff(row_slots), np.where(per_row > 1, per_row, 0))
    assert np.all(items[:, 2] <= chunk)
    cover = np.zeros(g.num_edges, np.int32)
    order_key = []
    next_slot = row_slots[:-1].copy()
    for r, b, c, slot in items:
        cover[b:b + c] += 1
        assert indptr[r] <= b and b + c <= indptr[r + 1]
        assert (slot >= 0) == (per_row[r] > 1)
        cb = int(indices[b] // col_block) if (col_block and c) else 0
        if col_block and c:
            assert int(indices[b + c - 1] // col_block) == cb      # an item never straddles column blocks
        order_key.append((cb, r, b))
    assert np.all(cover == 1)
    assert order_key == sorted(order_key)                         # (column block, row, position) order
    # slots of a row are consecutive and numbered in edge order
    multi = items[items[:, 3] >= 0]
    for r, b, c, slot in multi[np.lexsort((multi[:, 1], multi[:, 0]))]:
        assert slot == next_slot[r]
        next_slot[r] += 1
    assert np.array_equal(next_slot, np.where(per_row > 1, row_slots[1:], row_slots[:-1]))


@pytest.fixture(params=["simt", "tc"])
def gemm_mode(T, request):
    """Both realisations of COMP_MM: the FFMA kernel and the tcgen05 3xTF32 kernel."""
    T.k.set_gemm_mode(request.param)
    yield request.param
    T.k.set_gemm_mode("auto")


@pytest.mark.parametrize("n,k,f", [(2708, 1433, 128), (1000, 602, 128), (513, 128, 64), (300, 64, 16), (77, 500, 128),
                                   (260, 256, 256), (40000, 602, 128), (129, 7, 32), (1, 33, 48)])
def test_gemm_fp32(T, gemm_mode, n, k, f):
    rng = np.random.default_rng(n + k)
    x = rng.standard_normal((n, k), dtype=np.float32)
    w = synthetic.glorot(rng, k, f)
    xd = T.k.to_table(_dev(T, x))
    z = T.k.gemm(xd, _dev(T, w)).cpu().numpy()
    z64 = O.gemm(x, w)
    scale = np.abs(x).astype(np.float64) @ np.abs(w).astype(np.float64)
    assert_close_rowscale(z, z64, scale, what=f"gemm[{gemm_mode}] {n}x{k}x{f}")
    again = T.k.gemm(xd, _dev(T, w)).cpu().numpy()
    assert np.array_equal(z, again), "GEMM is not bitwise reproducible"


def test_gemm_tc_refuses_ineligible_shapes(T):
    T.k.set_gemm_mode("tc")
    try:
        x = T.k.to_table(_dev(T, np.ones((64, 40), np.float32)))
        with pytest.raises(T.cabi.GtaUnsupported):
            T.k.gemm(x, _dev(T, np.ones((40, 24), np.float32)))      # F not a multiple of 16
    finally:
        T.k.set_gemm_mode("auto")
    z = T.k.gemm(x, _dev(T, np.ones((40, 24), np.float32)))          # auto: falls back to FFMA
    assert float(z.min()) == 40.0 and float(z.max()) == 40.0


@pytest.mark.parametrize("heads", [1, 4, 8, 16])
def test_gemm_attention_projections(T, gemm_mode, heads):
    n, k, f = 700, 602, 128
    x, w, al, ar = synthetic.gat_tensors(n, k, f, heads, seed=3, dense_attention=(heads == 4))
    z, el, er = T.k.gemm(T.k.to_table(_dev(T, x)), _dev(T, w), _dev(T, al), _dev(T, ar))
    z64 = O.gemm(x, w)
    zs = np.abs(x).astype(np.float64) @ np.abs(w).astype(np.float64)
    assert_close_rowscale(z.cpu().numpy(), z64, zs, what="Z")
    assert_close_rowscale(el.cpu().numpy(), z64 @ al.astype(np.float64), zs @ np.abs(al).astype(np.float64), what="el")
    assert_close_rowscale(er.cpu().numpy(), z64 @ ar.astype(np.float64), zs @ np.abs(ar).astype(np.float64), what="er")


@pytest.mark.parametrize("name,n,e,seed,i0", GRAPHS)
@pytest.mark.parametrize("f", [16, 64, 128, 256, 500])
@pytest.mark.parametrize("chunk,col_block", [(32, 0), (1024, 0), (64, 500), (1024, 60)])
def test_aggregate_scalar_weight(T, name, n, e, seed, i0, f, chunk, col_block):
    g = _graph(name, n, e, seed, i0)
    indptr, indices, _ = O.csr_build(g.dst, g.src, n)
    dg = T.graph.csr_from_coo(g.dst, g.src, n)
    rng = np.random.default_rng(f)
    x = rng.standard_normal((n, f), dtype=np.float32)
    w = synthetic.gcn_edge_norm(indptr, indices)
    xd = T.k.to_table(_dev(T, x))
    got = T.k.aggregate(dg, xd, _dev(T, w), sched=dg.schedule(chunk, col_block)).cpu().numpy()
    want = O.spmm(indptr, indices, w, x)
    scale = O.spmm(indptr, indices, np.abs(w), np.abs(x))
    assert_close_rowscale(got, want, scale, what=f"aggregate f={f} chunk={chunk}")
    # plain gather ADD (no weights) and run-to-run bitwise reproducibility
    plain = T.k.aggregate(dg, xd, None, sched=dg.schedule(chunk, col_block))
    again = T.k.aggregate(dg, xd, None, sched=dg.schedule(chunk, col_block))
    assert T.torch.equal(plain, again)
    assert_close_rowscale(plain.cpu().numpy(), O.spmm(indptr, indices, None, x),
                          O.spmm(indptr, indices, None, np.abs(x)), what="plain gather")


@pytest.mark.parametrize("name,n,e,seed,i0", GRAPHS)
@pytest.mark.parametrize("f,heads", [(128, 4), (128, 8), (128, 16), (128, 1), (64, 4), (64, 16), (16, 4), (16, 2), (256, 8),
                                     # heads narrower than a 4-feature piece (layer 3 of the reference's GAT: F = H = 16)
                                     (16, 16), (16, 8), (8, 4), (8, 8), (32, 16), (4, 4), (4, 2), (64, 32)])
@pytest.mark.parametrize("chunk,col_block", [(32, 0), (1024, 0), (64, 500), (1024, 60)])
def test_gat_single_pass(T, name, n, e, seed, i0, f, heads, chunk, col_block):
    g = _graph(name, n, e, seed, i0)
    indptr, indices, _ = O.csr_build(g.dst, g.src, n)
    dg = T.graph.csr_from_coo(g.dst, g.src, n)
    x, w, al, ar = synthetic.gat_tensors(n, 96, f, heads, seed=seed)
    ref = O.gat_layer(indptr, indices, x, w, al, ar)
    z32 = ref["Z"].astype(np.float32)
    el32 = ref["el"].astype(np.float32)
    er32 = ref["er"].astype(np.float32)
    # oracle on the SAME fp32 inputs the kernel sees
    r2 = _gat_from_z(indptr, indices, z32, el32, er32)
    sched = dg.schedule(chunk, col_block)
    args = (dg, _dev(T, el32), _dev(T, er32), T.k.to_table(_dev(T, z32)))
    # want_stats tracks the true row maximum: the online-softmax path
    out, rowmax, rowsum = T.k.gat_aggregate(*args, sched=sched, want_stats=True)
    assert T.torch.equal(out, T.k.gat_aggregate(*args, sched=sched, bounded=False)), "online path not reproducible"
    # default: softmax shifted by the per-(row, column block) bound leaky(el + max er)
    out_b = T.k.gat_aggregate(*args, sched=sched)
    assert T.torch.equal(out_b, T.k.gat_aggregate(*args, sched=sched)), "bound path not bitwise reproducible"
    scale = O.gat_rowscale(indptr, indices, z32.astype(np.float64), r2["alpha"])
    assert_close_rowscale(out.cpu().numpy(), r2["Y"], scale, what=f"GAT online f={f} H={heads} chunk={chunk}")
    assert_close_rowscale(out_b.cpu().numpy(), r2["Y"], scale, what=f"GAT bound f={f} H={heads} chunk={chunk}")
    np.testing.assert_allclose(rowmax.cpu().numpy(), r2["rowmax"], rtol=1e-6, atol=1e-6)
    np.testing.assert_allclose(rowsum.cpu().numpy(), r2["S"], rtol=2e-5)


def test_er_stats_codes(T):
    """gta_er_stats: per column block and head, max er and max -er (ordered-int codes decode to the exact floats)."""
    rng = np.random.default_rng(5)
    er = (rng.standard_normal((1000, 4)) * 3).astype(np.float32)
    er[10, 2] = -0.0
    for col_block in (0, 256, 999):
        st = T.k.er_stats(_dev(T, er), col_block).cpu().numpy().view(np.uint32)
        blocks = 1 if col_block == 0 else -(-1000 // col_block)
        assert st.shape == (blocks, 2, 4)
        dec = np.where(st & 0x80000000, st & 0x7FFFFFFF, ~st).astype(np.uint32).view(np.float32)
        for b in range(blocks):
            lo, hi = (0, 1000) if col_block == 0 else (b * col_block, min((b + 1) * col_block, 1000))
            np.testing.assert_array_equal(dec[b, 0], er[lo:hi].max(axis=0))
            np.testing.assert_array_equal(-dec[b, 1], er[lo:hi].min(axis=0))
    assert T.k.er_stats(_dev(T, np.zeros((8, 3), np.float32))) is None          # 3 heads: no power of two


@pytest.mark.parametrize("heads,f", [(4, 128), (8, 128), (2, 16), (16, 16), (8, 16)])
@pytest.mark.parametrize("col_block", [0, 700])
def test_gat_bound_falls_back_when_the_er_range_is_wide(T, heads, f, col_block):
    """Source logits spanning far more than the bound path's exponent budget (60): those column blocks must take the
    online softmax; a narrow block beside a wide one keeps the bound.  Either way the result is the oracle's."""
    g = _graph("skew", 3000, 90000, 2, 3.0)
    n = g.num_nodes
    indptr, indices, _ = O.csr_build(g.dst, g.src, n)
    dg = T.graph.csr_from_coo(g.dst, g.src, n)
    rng = np.random.default_rng(7)
    z = rng.standard_normal((n, f), dtype=np.float32)
    el = rng.standard_normal((n, heads), dtype=np.float32)
    er = rng.standard_normal((n, heads), dtype=np.float32)
    er[:700] *= 80.0          # the first column block (or the whole table) spans about +-300
    r = _gat_from_z(indptr, indices, z, el, er)
    sched = dg.schedule(1024, col_block)
    out = T.k.gat_aggregate(dg, _dev(T, el), _dev(T, er), T.k.to_table(_dev(T, z)), sched=sched)
    assert T.torch.equal(out, T.k.gat_aggregate(dg, _dev(T, el), _dev(T, er), T.k.to_table(_dev(T, z)), sched=sched))
    scale = O.gat_rowscale(indptr, indices, z.astype(np.float64), r["alpha"])
    assert_close_rowscale(out.cpu().numpy(), r["Y"], scale, what=f"wide er range H={heads} col_block={col_block}")


def _gat_from_z(indptr, indices, z, el, er):
    """Oracle edge phase on given (fp32-rounded) Z, el, er, evaluated in fp64."""
    rows = O.row_ids(indptr)
    z, el, er = z.astype(np.float64), el.astype(np.float64), er.astype(np.float64)
    lr = O.leaky_relu(el[rows] + er[indices])
    mx = O.segment_max(lr, indptr)
    mx = np.where(np.isfinite(mx), mx, 0)
    p = np.exp(lr - mx[rows])
    s = O.segment_sum(p, indptr)
    alpha = p / s[rows]
    o = O.segment_sum(O.head_broadcast(alpha, z.shape[1]) * z[indices], indptr)
    return {"p": p, "S": s, "rowmax": mx, "alpha": alpha, "O": o, "Y": O.elu(o)}


@pytest.mark.parametrize("heads,f", [(4, 128), (16, 128), (4, 64), (16, 64), (8, 64), (2, 16)])
def test_gat_two_block_path(T, heads, f):
    """ISA blocks [4,5,6,7,8] then [3,9,10,11,12,13] as separate kernels (STORE_E p honoured)."""
    g = _graph("skew", 3000, 90000, 2, 3.0)
    n = g.num_nodes
    indptr, indices, _ = O.csr_build(g.dst, g.src, n)
    dg = T.graph.csr_from_coo(g.dst, g.src, n)
    rng = np.random.default_rng(1)
    z = rng.standard_normal((n, f), dtype=np.float32)
    el = rng.standard_normal((n, heads), dtype=np.float32)
    er = rng.standard_normal((n, heads), dtype=np.float32)
    r = _gat_from_z(indptr, indices, z, el, er)
    p, rowmax, rowsum = T.k.gat_logits(dg, _dev(T, el), _dev(T, er))
    np.testing.assert_allclose(p.cpu().numpy(), r["p"], rtol=2e-6, atol=1e-30)
    np.testing.assert_allclose(rowsum.cpu().numpy(), r["S"], rtol=2e-5)
    out = T.k.aggregate(dg, T.k.to_table(_dev(T, z)), p, rowden=rowsum, epilogue=T.cabi.EPI_ELU)
    scale = O.gat_rowscale(indptr, indices, z.astype(np.float64), r["alpha"])
    assert_close_rowscale(out.cpu().numpy(), r["Y"], scale, rtol=2e-5, what="two-block GAT")


@pytest.mark.parametrize("name,n,e,seed,i0", GRAPHS)
@pytest.mark.parametrize("f", [16, 6, 128, 256])
@pytest.mark.parametrize("terms,unary", [("exr", "relu"), ("exr", "elu"), ("exr", "copy"), ("xr", "relu"), ("e", "relu"),
                                         ("x", "copy"), ("er", "relu"), ("ex", "elu")])
@pytest.mark.parametrize("chunk,col_block", [(32, 0), (1024, 60)])
def test_edge_sum_single_pass(T, name, n, e, seed, i0, f, terms, unary, chunk, col_block):
    """gta_aggregate_edge_sum_f32 (PNA ops 5-8): out[i] = sum_k unary(edge[k] + x[src k] + rowterm[i]) against fp64."""
    g = _graph(name, n, e, seed, i0)
    indptr, indices, _ = O.csr_build(g.dst, g.src, n)
    rows = O.row_ids(indptr)
    dg = T.graph.csr_from_coo(g.dst, g.src, n)
    rng = np.random.default_rng(seed + f)
    edge = rng.standard_normal((len(indices), f), dtype=np.float32) if "e" in terms else None
    x = rng.standard_normal((n, f), dtype=np.float32) if "x" in terms else None
    r = rng.standard_normal((n, f), dtype=np.float32) if "r" in terms else None
    v = np.zeros((len(indices), f))
    sc = np.zeros((len(indices), f))
    for t, sel in ((edge, slice(None)), (x, indices), (r, rows)):
        if t is not None:
            v = v + t[sel].astype(np.float64)
            sc = sc + np.abs(t[sel]).astype(np.float64)
    y64 = O.segment_sum({"relu": lambda a: np.maximum(a, 0), "elu": O.elu, "copy": lambda a: a}[unary](v), indptr)
    scale = O.segment_sum(sc, indptr)
    code = {"relu": T.cabi.UN_RELU, "elu": T.cabi.UN_ELU, "copy": T.cabi.UN_COPY}[unary]
    tab = lambda a: None if a is None else T.k.to_table(_dev(T, a))
    sched = dg.schedule(chunk, col_block)
    out = T.k.aggregate_edge_sum(dg, tab(edge), tab(x), tab(r), code, sched=sched)
    assert out.shape == (n, f)
    assert T.torch.equal(out, T.k.aggregate_edge_sum(dg, tab(edge), tab(x), tab(r), code, sched=sched)), "not reproducible"
    assert_close_rowscale(out.cpu().numpy(), y64, scale, what=f"edge sum {terms} {unary} f={f} chunk={chunk}")
    # with an applynode epilogue on top
    out_e = T.k.aggregate_edge_sum(dg, tab(edge), tab(x), tab(r), code, epilogue=T.cabi.EPI_RELU, sched=sched)
    assert_close_rowscale(out_e.cpu().numpy(), np.maximum(y64, 0), scale, what="edge sum + ReLU epilogue")


@pytest.mark.parametrize("chunk,col_block", [(32, 0)])
def test_static_striding_is_the_same_reduction(T, monkeypatch, chunk, col_block):
    """GTA_PHASE_STATIC (long lists of tiny items, the RMAT shapes: warps stride through the work list instead of
    taking items from the counter) only changes WHO runs an item, never the reduction: every kernel must return the
    bits of the dynamic launch.  Forced here on a small graph by lowering the thresholds of kernels._launch_blocks."""
    # the library strides statically only when a warp gets at least 32 steps (aggregate_common.cuh take_for): with up to 5 920
    # resident warps that takes 190 k items -- 400 k rows of about 6 edges give one or more items per row
    g = synthetic.powerlaw_graph(400_000, 2_400_000, seed=3, i0=50.0, name="wide-low-degree")
    n = g.num_nodes
    dg = T.graph.csr_from_coo(g.dst, g.src, n)
    sched = dg.schedule(chunk, col_block)
    assert sched.num_items >= 32 * 5920
    rng = np.random.default_rng(11)
    z = T.k.to_table(_dev(T, rng.standard_normal((n, 128), dtype=np.float32)))
    z256 = T.k.to_table(_dev(T, rng.standard_normal((n, 256), dtype=np.float32)))
    zb = T.k.to_table(z.to(T.torch.bfloat16))
    el, er = _dev(T, rng.standard_normal((n, 4), dtype=np.float32)), _dev(T, rng.standard_normal((n, 4), dtype=np.float32))
    el16, er16 = _dev(T, rng.standard_normal((n, 16), dtype=np.float32)), _dev(T, rng.standard_normal((n, 16), dtype=np.float32))
    w = _dev(T, rng.random((g.num_edges, 1), dtype=np.float32))
    et = T.k.to_table(_dev(T, rng.standard_normal((g.num_edges, 128), dtype=np.float32)))
    # widths just above one feature window: every kernel then runs a second window (blockIdx.y = 1) of the same cursor
    gen = T.torch.Generator(device="cuda").manual_seed(12)
    zw = T.torch.randn((n, 260), generator=gen, device="cuda")
    el2, er2, el12, er12 = (T.torch.randn((n, h), generator=gen, device="cuda") for h in (2, 2, 12, 12))
    w3 = T.torch.rand((g.num_edges, 3), generator=gen, device="cuda") + 0.1
    runs = {
        "aggregate": lambda: T.k.aggregate(dg, z, w, sched=sched),
        "aggregate 256 wide": lambda: T.k.aggregate(dg, z256, w, sched=sched),
        "aggregate bf16": lambda: T.k.aggregate(dg, zb, w, sched=sched),
        "gat": lambda: T.k.gat_aggregate(dg, el, er, z, sched=sched),
        "gat online": lambda: T.k.gat_aggregate(dg, el, er, z, sched=sched, bounded=False),
        "gat bf16": lambda: T.k.gat_aggregate(dg, el, er, zb, sched=sched),
        "gat 16 heads": lambda: T.k.gat_aggregate(dg, el16, er16, z, sched=sched),
        "edge sum": lambda: T.k.aggregate_edge_sum(dg, et, z, z, T.cabi.UN_RELU, sched=sched),
        "aggregate 260 wide unweighted": lambda: T.k.aggregate(dg, zw, sched=sched),
        "aggregate 132 wide per-head": lambda: T.k.aggregate(dg, zw[:, :132], w3, sched=sched),
        "gat 136 wide 2 heads": lambda: T.k.gat_aggregate(dg, el2, er2, zw[:, :136], sched=sched),
        "gat 144 wide 12 heads": lambda: T.k.gat_aggregate(dg, el12, er12, zw[:, :144], sched=sched),
    }
    dynamic = {k: f().clone() for k, f in runs.items()}
    monkeypatch.setattr(T.k, "STATIC_MIN_ITEMS", 0)
    monkeypatch.setattr(T.k, "STATIC_ITEM_EDGES", 1 << 30)
    for k, f in runs.items():
        assert T.torch.equal(f(), dynamic[k]), f"{k}: static striding changed the result"


def test_generic_edge_and_node_ops(T):
    g = _graph("tiny", 64, 300, 1, 5.0)
    n = g.num_nodes
    indptr, indices, _ = O.csr_build(g.dst, g.src, n)
    rows = O.row_ids(indptr)
    dg = T.graph.csr_from_coo(g.dst, g.src, n)
    rng = np.random.default_rng(0)
    a = rng.standard_normal((n, 4), dtype=np.float32)
    b = rng.standard_normal((n, 4), dtype=np.float32)
    zt = rng.standard_normal((n, 32), dtype=np.float32)
    C = T.cabi
    s = T.k.edge_binary(dg, C.BIN_ADD, _dev(T, a), C.OPND_DST, _dev(T, b), C.OPND_SRC)
    np.testing.assert_array_equal(s.cpu().numpy(), a[rows] + b[indices])
    p = T.k.edge_unary(dg, C.UN_EXP_LEAKY_RELU, s, C.OPND_EDGE)
    np.testing.assert_allclose(p.cpu().numpy(), np.exp(O.leaky_relu(a[rows] + b[indices])), rtol=1e-6)
    m = T.k.edge_binary(dg, C.BIN_MUL, p, C.OPND_EDGE, _dev(T, zt), C.OPND_SRC)
    np.testing.assert_allclose(m.cpu().numpy(), np.repeat(p.cpu().numpy(), 8, axis=1) * zt[indices], rtol=1e-6)
    zs = T.k.edge_unary(dg, C.UN_COPY, _dev(T, zt), C.OPND_SRC)
    np.testing.assert_array_equal(zs.cpu().numpy(), zt[indices])
    q = T.k.node_binary(C.BIN_DIV, _dev(T, zt), _dev(T, np.abs(a) + 1))
    np.testing.assert_allclose(q.cpu().numpy(), zt / np.repeat(np.abs(a) + 1, 8, axis=1), rtol=1e-6)
    e = T.k.node_unary(C.UN_ELU, _dev(T, zt))
    np.testing.assert_allclose(e.cpu().numpy(), O.elu(zt), rtol=1e-6, atol=1e-7)


def test_errors_are_loud(T):
    g = _graph("tiny", 64, 300, 1, 5.0)
    dg = T.graph.csr_from_coo(g.dst, g.src, g.num_nodes)
    x = T.torch.zeros((64, 6), device="cuda")           # width not a multiple of 4
    with pytest.raises(T.cabi.GtaError):
        T.k.aggregate(dg, x)
    with pytest.raises(T.cabi.GtaUnsupported):            # per-head width 3: neither whole pieces nor 2 nor 1
        T.k.gat_aggregate(dg, T.torch.zeros((64, 4), device="cuda"), T.torch.zeros((64, 4), device="cuda"),
                          T.torch.zeros((64, 12), device="cuda"))
    with pytest.raises(T.cabi.GtaUnsupported):            # narrow heads on a bf16 table have no kernel
        T.k.gat_aggregate(dg, T.torch.zeros((64, 8), device="cuda"), T.torch.zeros((64, 8), device="cuda"),
                          T.k.to_table(T.torch.zeros((64, 16), device="cuda", dtype=T.torch.bfloat16)))
    with pytest.raises(RuntimeError):
        T.k.aggregate(dg, T.torch.zeros((64, 8)))          # CPU tensor: no CPU fallback


def test_tile_table_files_match_the_reference_byte_for_byte(T, golden_dir, tmp_path):
    """graph.write_tile_tables writes what code/preprocessing.py's CLI writes (adj_<ds>_<SR>_1.yaml,
    sizelist, maxlist) -- compared with the files the unmodified reference produced."""
    import os
    z = np.load(os.path.join(golden_dir, "tiles", "g97.npz"))
    n = int(z["num_nodes"])
    dg = T.graph.csr_from_coo(z["dst"], z["src"], n)
    sizes = sorted(int(k.split("_")[1]) for k in z.files if k.startswith("table_"))
    T.graph.write_tile_tables(dg, "g97", sizes, root=str(tmp_path))
    names = [f"adj_g97_{sr}_1.yaml" for sr in sizes] + ["sizelist_g97.yaml", "maxlist_g97.yaml"]
    for name in names:
        want = open(os.path.join(golden_dir, "tiles", name), "rb").read()
        got = open(os.path.join(str(tmp_path), "dataset", "g97", name), "rb").read()
        assert got == want, name


def test_divided_weights_next_to_an_empty_row(T):
    """Two rows share a warp when F <= 64; an EMPTY row (rowden = 0) beside a non-empty one must stay 0,
    not 0/0 (regression: GAT layer 2 with STORE_* honoured)."""
    n, f, h = 8, 64, 16
    dst = np.array([1, 1, 1, 3, 3], dtype=np.int32)      # rows 0, 2, 4..7 have no edges
    src = np.array([0, 2, 5, 1, 7], dtype=np.int32)
    dg = T.graph.csr_from_coo(dst, src, n)
    rng = np.random.default_rng(0)
    z = rng.standard_normal((n, f), dtype=np.float32)
    el = rng.standard_normal((n, h), dtype=np.float32)
    er = rng.standard_normal((n, h), dtype=np.float32)
    p, _, rowsum = T.k.gat_logits(dg, _dev(T, el), _dev(T, er))
    out = T.k.aggregate(dg, T.k.to_table(_dev(T, z)), p, rowden=rowsum, epilogue=T.cabi.EPI_ELU).cpu().numpy()
    assert np.all(np.isfinite(out))
    assert np.all(out[[0, 2, 4, 5, 6, 7]] == 0)
    scalar = T.k.aggregate(dg, T.k.to_table(_dev(T, z)), p[:, :1].contiguous(), rowden=rowsum[:, :1].contiguous()).cpu().numpy()
    assert np.all(np.isfinite(scalar)) and np.all(scalar[[0, 2, 4, 5, 6, 7]] == 0)
