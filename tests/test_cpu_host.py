"""Host logic that needs no GPU: ISA loader on every golden program, block/op attribution,
the C-ABI library's exported symbols, and failure modes."""
import ctypes
import json
import os
import re

import pytest
import yaml

from gta_graph_tensor_acclelrator_for_general_gnn_b200 import _cabi, isa

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(REPO, "tests", "golden")
with open(os.path.join(GOLDEN, "manifest.json")) as _f:
    MANIFEST = json.load(_f)


def _load(rel):
    with open(os.path.join(GOLDEN, rel)) as f:
        return yaml.safe_load(f)


@pytest.mark.parametrize("prog", MANIFEST["programs"], ids=[p["file"].split("/")[-1][:-5] for p in MANIFEST["programs"]])
def test_program_loads_and_blocks_match_the_plan(prog):
    program = isa.Program.from_records(_load(prog["file"]))
    op_info = _load(prog["opgraph"])
    assert len(program.blocks) == len(prog["op_array"])
    # the op sets recovered from the instruction stream alone equal the plan interpret() was given
    assert [sorted(b) for b in program.block_ops(op_info)] == [sorted(b) for b in prog["op_array"]]
    for block in program.blocks:
        for inst in block:
            assert inst.type != "FETCH"
            assert inst.tile_times > 0 and inst.tile_size > 0 and inst.feature_length > 0
            for _, dep_id, times in inst.raw + inst.war:
                isa.parse_id(dep_id)
                assert len(times) == 2


def test_fused_instruction_is_recognised():
    prog = next(p for p in MANIFEST["programs"] if p["file"].endswith("GCN-flickr-layer1-trans__0_1-2-3.yaml"))
    program = isa.Program.from_records(_load(prog["file"]))
    fused = [i for i in program.blocks[1] if i.type == "COMP_MUL_COMP_ADD"]
    assert len(fused) == 1
    assert fused[0].comp_types == ("MUL", "ADD")
    assert [(r.op, r.kind) for r in fused[0].refs] == [(2, "applyedge"), (3, "gather")]
    assert fused[0].tile_times == 175 * 89250           # TR*TC, SURVEY Appendix B1
    assert program.stored_ops() == [[0], [3]]


def test_loader_rejects_garbage():
    with pytest.raises(isa.IsaError):
        isa.Program.from_records({"not": "a list"})
    with pytest.raises(isa.IsaError):
        isa.Program.from_records([[{"TYPE": "COMP_MM"}]])
    good = _load(MANIFEST["programs"][0]["file"])
    with pytest.raises(isa.IsaError):
        isa.Program.from_records([[dict(good[0][0], TYPE="FETCH")]])
    with pytest.raises(isa.IsaError):
        isa.Program.from_records([[dict(good[0][0], ID="0_bogus_0")]])


def test_library_exports_every_declared_symbol():
    """include/gta_b200.h <-> _cabi.SIGNATURES <-> libgta_b200.so agree (no compute calls)."""
    header = open(os.path.join(REPO, "include", "gta_b200.h")).read()
    declared = set(re.findall(r"\b(gta_[a-z0-9_]+)\s*\(", header))
    assert declared == set(_cabi.SIGNATURES), declared ^ set(_cabi.SIGNATURES)
    if not os.path.exists(_cabi.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    lib = _cabi.load()
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.gta_abi_version() == 1
    assert lib.gta_schedule_max_items(10, 100, 32, 10, 0) == 14
    assert lib.gta_schedule_max_items(10, 100, 32, 10, 3) == 44      # 4 column blocks
    assert lib.gta_gat_partial_stride(128, 4) == 136 and lib.gta_gat_partial_stride(16, 1) == 20


def test_missing_library_fails_loudly(monkeypatch, tmp_path):
    monkeypatch.setattr(_cabi, "_lib", None)
    monkeypatch.setattr(_cabi, "LIB_PATH", str(tmp_path / "nope.so"))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        _cabi.load()


def test_cpu_tensors_are_refused():
    import numpy as np
    import torch
    from gta_graph_tensor_acclelrator_for_general_gnn_b200 import graph
    if torch.cuda.is_available():
        pytest.skip("CPU-only check")
    with pytest.raises(RuntimeError):
        graph.csr_from_coo(torch.zeros(4, dtype=torch.int32), torch.zeros(4, dtype=torch.int32), 4)
    with pytest.raises((RuntimeError, AssertionError)):
        graph.csr_from_coo(np.zeros(4, np.int32), np.zeros(4, np.int32), 4)   # upload needs a GPU


def test_read_csr_npz_expands_to_coo_and_rejects_bad_archives(tmp_path):
    """Host half of the SciPy-CSR .npz ingest (the format simulator.py:74-84 reads)."""
    import numpy as np
    import scipy.sparse as sp
    from gta_graph_tensor_acclelrator_for_general_gnn_b200 import graph
    rng = np.random.default_rng(3)
    a = sp.random(40, 40, density=0.1, random_state=7, format="csr", dtype=np.float32)
    p = tmp_path / "adj.npz"
    sp.save_npz(p, a)
    dst, src, data, n = graph.read_csr_npz(str(p))
    coo = a.tocoo()
    assert n == 40 and dst.dtype == np.int32 and src.dtype == np.int32
    assert np.array_equal(dst, coo.row) and np.array_equal(src, coo.col) and np.array_equal(data, coo.data)
    np.savez(tmp_path / "nokeys.npz", indices=a.indices, indptr=a.indptr)
    with pytest.raises(KeyError, match="required keys"):
        graph.read_csr_npz(str(tmp_path / "nokeys.npz"))
    np.savez(tmp_path / "rect.npz", data=a.data, indices=a.indices, indptr=a.indptr, shape=np.array([40, 41]))
    with pytest.raises(ValueError, match="square"):
        graph.read_csr_npz(str(tmp_path / "rect.npz"))
    np.savez(tmp_path / "short.npz", data=a.data, indices=a.indices, indptr=a.indptr[:-1], shape=np.array([40, 40]))
    with pytest.raises(ValueError, match="inconsistent"):
        graph.read_csr_npz(str(tmp_path / "short.npz"))
    bad = a.indices.copy()
    bad[0] = 40
    np.savez(tmp_path / "oob.npz", data=a.data, indices=bad, indptr=a.indptr, shape=np.array([40, 40]))
    with pytest.raises(ValueError, match="outside"):
        graph.read_csr_npz(str(tmp_path / "oob.npz"))
    empty = sp.csr_matrix((5, 5), dtype=np.float32)
    sp.save_npz(tmp_path / "empty.npz", empty)
    dst, src, data, n = graph.read_csr_npz(str(tmp_path / "empty.npz"))
    assert n == 5 and dst.size == src.size == data.size == 0


def test_ctypes_signatures_match_the_header_prototypes():
    """Every parameter of every prototype in include/gta_b200.h has the width/kind its ctypes binding
    declares (an int32/int64 or pointer/scalar mismatch would corrupt arguments silently)."""
    import ctypes as C
    header = open(os.path.join(REPO, "include", "gta_b200.h")).read()
    header = re.sub(r"/\*.*?\*/", " ", header, flags=re.S)
    header = re.sub(r"//[^\n]*", " ", header)
    protos = re.findall(r"([A-Za-z_][A-Za-z0-9_ \*]*?)\b(gta_[a-z0-9_]+)\s*\(([^()]*)\)\s*;", header)
    assert {name for _, name, _ in protos} == set(_cabi.SIGNATURES)

    def kind(ctype):
        if ctype is None:
            return "void"
        if ctype in (C.c_void_p, C.c_char_p) or isinstance(ctype, type) and issubclass(ctype, C._Pointer):
            return "ptr"
        if ctype is C.c_float:
            return "f32"
        return {4: "i32", 8: "i64"}[C.sizeof(ctype)] if ctype is not C.c_size_t else "size"

    def ckind(text):
        text = re.sub(r"\bconst\b", "", text).strip()
        if "*" in text:
            return "ptr"
        base = text.split()[0] if len(text.split()) > 1 or text in ("void", "int") else text
        return {"void": "void", "int": "i32", "int32_t": "i32", "int64_t": "i64", "size_t": "size", "float": "f32",
                "uint32_t": "i32", "uint64_t": "i64"}[base]

    for ret, name, params in protos:
        res, args = _cabi.SIGNATURES[name]
        ret = re.sub(r"\b(extern|GTA_API)\b", "", ret).strip()
        assert ckind(ret + " r") == kind(res), (name, "return", ret)
        plist = [p.strip() for p in params.split(",") if p.strip() and p.strip() != "void"]
        assert len(plist) == len(args), (name, len(plist), len(args))
        for i, (ptext, ctype) in enumerate(zip(plist, args)):
            assert ckind(ptext) == kind(ctype), (name, i, ptext, ctype)


def test_model_times_fixture_refers_to_golden_programs():
    """tests/golden/model_times.json (the reference simulator's modelled latency, oracle/gen_model_times.py)
    names only programs of the manifest, and every entry is either a result or a recorded failure."""
    import json
    with open(os.path.join(GOLDEN, "model_times.json")) as f:
        model = json.load(f)
    files = {p["file"] for p in MANIFEST["programs"] if p["dataset"] == "cora"}
    assert {m["file"] for m in model["programs"]} == files
    done = [m for m in model["programs"] if "cycles" in m]
    assert len(done) >= 10 and all(m["cycles"] > 0 and m["rw_bytes"] > 0 for m in done)
    assert all("error" in m for m in model["programs"] if "cycles" not in m)
    # known-answer anchor from the reference's own record of this plan family: the fused 3-block GAT plan is
    # modelled faster than the unfused one
    by = {m["file"].split("/")[-1]: m for m in done}
    assert by["GAT-cora-layer1-original__0-1-2_4-5-6-7-8_3-9-10-11-12-13.yaml"]["cycles"] < \
        by["GAT-cora-layer1-original__0_1_2_3_4_5_6_7_8_9_10_11_12_13.yaml"]["cycles"]


def test_c_abi_rejects_bad_arguments_without_a_gpu():
    """Every entry point validates its arguments before it touches the device: null pointers and impossible
    sizes come back as GTA_ERR_INVALID with a message naming the function (no launch, so this runs on CPU)."""
    lib = _cabi.load()

    def refused(name, rc):
        assert rc == _cabi.ERR_INVALID, (name, rc)
        assert lib.gta_last_error().decode().startswith(name), (name, lib.gta_last_error())

    n = None
    refused("gta_csr_build", lib.gta_csr_build(n, n, 10, 5, n, n, n, n, 0, n))
    refused("gta_csr_build", lib.gta_csr_build(n, n, -1, 5, n, n, n, n, 0, n))
    refused("gta_tile_nnz", lib.gta_tile_nnz(n, n, 10, 0, 0, 1, n, n))
    refused("gta_partition", lib.gta_partition(n, 10, 0, n, n))
    refused("gta_gemm_f32", lib.gta_gemm_f32(n, 0, n, 0, n, 0, 10, 4, 4, n, n, 0, n, n, 0, n, 0, n))
    refused("gta_aggregate_f32", lib.gta_aggregate_f32(n, 1, n, 0, n, 0, n, 0, n, n, 4, n, 4, 4, 0, n, n, n, 3, n))
    refused("gta_gat_aggregate_f32", lib.gta_gat_aggregate_f32(n, 1, n, 0, n, n, n, 4, 4, 0.2, n, 128, n, 128, 128, 0,
                                                              n, n, n, n, n, 0, n, 3, n))
    refused("gta_er_stats", lib.gta_er_stats(n, 4, 10, 0, 4, n, n))
    refused("gta_edge_binary_f32", lib.gta_edge_binary_f32(n, n, 0, 1, 0, n, 0, 3, 3, n, 0, 4, 4, n, 4, 4, n))
    refused("gta_node_unary_f32", lib.gta_node_unary_f32(9, 0.2, n, 4, n, 4, 4, 1, n))
    refused("gta_schedule_build", lib.gta_schedule_build(n, n, 0, 1, 1, 0, 0, n, 0, n, n, n, n, 0, n))
    refused("gta_exchange_publish", lib.gta_exchange_publish(n, 0, 0, 99, 1, n, n))
    assert lib.gta_exchange_signal_bytes() >= 64 + 2 * 16 * 64 * 4
    refused("gta_gemm_set_mode", lib.gta_gemm_set_mode(7))
    assert lib.gta_gemm_get_mode() in (0, 1, 2)


def test_bench_reference_arm_prints_one_contract_line():
    """`bench.py --impl reference` (the CPU arm the driver runs beside the GPU arm): exactly one JSON line on stdout
    with the contract's keys, on a small workload so the CPU suite stays fast."""
    import json
    import subprocess
    import sys
    out = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--impl", "reference", "--workload", "cora-gat",
                          "--steps", "3", "--warmup", "3"], capture_output=True, text=True, timeout=600, check=True).stdout
    lines = [l for l in out.splitlines() if l.strip()]
    assert len(lines) == 1, out
    line = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert key in line, key
    assert line["impl"] == "reference" and line["unit"] == "GTEPS" and line["higher_is_better"] is True
    assert line["value"] > 0 and line["steps"] == 3 and line["vs_baseline"] is None and line["gpu_launches"] == 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1 and line["cpu_baseline"]["sample"]
    assert line["e2e"] == {"value": line["value"], "unit": "GTEPS", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in line["config"] and "model" not in line["config"]


def test_bench_refuses_to_run_the_gpu_arm_without_a_gpu():
    import subprocess
    import sys
    import torch
    if torch.cuda.is_available():
        pytest.skip("CPU-only check")
    r = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--workload", "cora-gat", "--steps", "1"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode != 0 and "no CPU fallback" in (r.stderr + r.stdout)


def _bench_module():
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(REPO, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


@pytest.mark.parametrize("rows,cols", [(300, 128), (232965, 128), (1 << 16, 256)])
def test_bench_dump_outputs_stays_in_budget_and_samples_the_same_rows(rows, cols, tmp_path):
    """--dump-outputs: every row when they fit 64 MB, else the same seeded row sample on every call; values are the
    rows the ids name (offset by the rank's first row)."""
    import numpy as np
    import torch
    bench = _bench_module()
    y = torch.arange(rows * cols, dtype=torch.float32).reshape(rows, cols) % 1021
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), y, 7)
    assert sum(os.path.getsize(p) for p in tmp_path.glob("a/*")) <= 64 * 10**6
    vals, ids = np.load(tmp_path / "a" / "output.npy"), np.load(tmp_path / "a" / "output_rows.npy")
    assert vals.dtype == np.float32 and ids.dtype == np.float64 and vals.shape[1] == cols
    assert np.array_equal(vals, y.numpy()[ids.astype(np.int64) - 7])
    assert np.all(np.diff(ids) > 0) and (vals.shape[0] == rows) == (rows * (cols * 4 + 8) <= 64 * 10**6 - 4096)
    assert np.array_equal(ids, np.load(tmp_path / "b" / "output_rows.npy"))
    assert np.array_equal(vals, np.load(tmp_path / "b" / "output.npy"))


@pytest.mark.gpu
def test_bench_dump_outputs_writes_the_benchmarked_layer(tmp_path):
    """bench.py --dump-outputs on the Cora GAT layer: the whole output (2708 x 128, rows 0..N-1) equals the fp64
    oracle's GAT layer on the bench's seeded inputs, within the fp32 error scale smoke() uses."""
    import subprocess
    import sys
    import numpy as np
    from oracle import gta_oracle as O
    from gta_graph_tensor_acclelrator_for_general_gnn_b200 import synthetic
    subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--workload", "cora-gat", "--steps", "2",
                    "--warmup", "3", "--no-e2e", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                   capture_output=True, text=True, timeout=600, check=True)
    vals, ids = np.load(tmp_path / "output.npy"), np.load(tmp_path / "output_rows.npy")
    n, _, fin = synthetic.SHAPES["cora"]
    assert vals.shape == (n, 128) and vals.dtype == np.float32 and np.all(np.isfinite(vals))
    assert np.array_equal(ids, np.arange(n, dtype=np.float64))
    g = synthetic.shape_graph("cora")
    x, w, al, ar = synthetic.gat_tensors(n, fin, 128, 4, seed=0)
    indptr, indices, _ = O.csr_build(g.dst, g.src, n)
    ref = O.gat_layer(indptr, indices, x, w, al, ar)
    zscale = np.abs(x).astype(np.float64) @ np.abs(w).astype(np.float64)
    scale = O.segment_sum(O.head_broadcast(ref["alpha"], 128) * zscale[indices], indptr)
    err = np.abs(vals - ref["Y"]) / (1e-5 * np.abs(ref["Y"]) + 1e-5 * scale + 1e-30)
    assert err.max() <= 1.0, f"dumped output {err.max():.2f}x the tolerance away from the fp64 oracle"


@pytest.mark.parametrize("n", [1, 2, 4, 8])
def test_committed_bench_lines_carry_the_contract_keys(n):
    """profiles/r01_bench_n*.json: the GPU arm's lines as measured on the box (what DESIGN.md quotes)."""
    import json
    with open(os.path.join(REPO, "profiles", f"r01_bench_n{n}.json")) as f:
        line = json.loads([l for l in f.read().splitlines() if l.startswith("{")][-1])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "clocks", "e2e", "gpu_launches", "roofline"):
        assert key in line, key
    assert line["n_gpus"] == n and line["warmup"] >= 3 and line["gpu_launches"] > 0 and line["dtype"] == "f32"
    assert abs(line["value"] - 114615892 / (line["ms_per_step"] * 1e-3) / 1e9) < 1e-6 * line["value"]
    roof = line["roofline"]
    assert roof["bound"] == "hbm" and roof["unit"] == "GB/s" and abs(roof["frac"] - roof["achieved"] / roof["peak"]) < 1e-9
    e2e = line["e2e"]
    assert e2e["h2d_bytes_per_step"] > 0 and e2e["d2h_bytes_per_step"] > 0 and 0 < e2e["value"] < line["value"] * 1.5
    assert not set(line["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
    if n == 1:
        assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["value"] > 0


@pytest.mark.parametrize("name,n,workload_edges", [
    ("r02_bench_n1", 1, 114615892), ("r02_bench_n2_fused", 2, 114615892), ("r02_bench_n1_reddit_gcn", 1, 114615892),
    ("r02_bench_n1_bf16", 1, 114615892), ("r02_bench_n1_reddit_heavy_gat", 1, 114615892),
])
def test_round2_bench_lines_carry_parity_and_the_measured_ceilings(name, n, workload_edges):
    """profiles/r02_bench_*.json (what DESIGN.md quotes for round 2): the contract keys, plus the round-2 additions --
    a parity object over the benchmarked output that is inside the tolerance and bitwise reproducible, the measured
    L2 gather ceiling next to the HBM roofline, the H2D floor next to the end-to-end number."""
    import json
    with open(os.path.join(REPO, "profiles", name + ".json")) as f:
        line = json.loads([l for l in f.read().splitlines() if l.startswith("{")][-1])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "clocks", "e2e", "gpu_launches", "roofline", "parity"):
        assert key in line, key
    assert line["n_gpus"] == n and line["warmup"] >= 3 and line["gpu_launches"] > 0 and line["vs_baseline"] is None
    assert abs(line["value"] - workload_edges / (line["ms_per_step"] * 1e-3) / 1e9) < 1e-6 * line["value"]
    par = line["parity"]
    assert par["max_err_over_tol"] <= 1.0 and par["bitwise_rerun"] is True and par["finite"] is True
    assert par["rows"] > 0 and par["edges"] > 0 and par["rows"] <= par["rows_of"]
    roof = line["roofline"]
    assert roof["bound"] == "hbm" and abs(roof["frac"] - roof["achieved"] / roof["peak"]) < 1e-9
    assert roof["l2_gather_peak_gbs"] > roof["peak"] and 0 < roof["l2_frac"] < 1.2
    assert (roof["traffic"] is None) == (n > 1 or "no ncu capture" in roof["traffic_source"])
    assert not set(line["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
    if line["e2e"] is not None:
        e2e = line["e2e"]
        assert e2e["h2d_bytes_per_step"] > 0 and e2e["d2h_bytes_per_step"] > 0 and 0 < e2e["value"] < line["value"]
        assert e2e["h2d_alone_ms"] <= e2e["ms_per_step"] * 1.02          # a step cannot beat its own upload


def test_item_size_and_slot_groups_are_functions_of_the_shape_only():
    """auto_chunk / slot_groups decide the reduction SHAPE: pure functions, so results stay bitwise reproducible."""
    from gta_graph_tensor_acclelrator_for_general_gnn_b200 import dist as gdist, graph
    assert [graph.auto_chunk(e) for e in (10556, 14_300_000, 57_300_000, 114_615_892, 268_435_456)] == [1024] * 5
    for world in range(1, 17):
        groups = gdist.slot_groups(world)
        assert groups[0] == [0] and [k for g in groups for k in g] == list(range(world)) and len(groups) <= 3


def test_built_library_holds_the_blackwell_instructions_the_design_claims():
    """Static check of the in-tree libgta_b200.so (no GPU): the GEMM is tcgen05 + TMA + TMEM, the aggregation kernels
    carry the in-launch exchange (system-scope peer loads and signal stores) and the cp.async item staging -- what
    DESIGN.md sections 4-5 state and tools/static_evidence.sh prints in full.  A build that silently lost one of
    these (a fallback path, a dropped -gencode) fails here, before any GPU time is spent."""
    import shutil
    import subprocess
    from gta_graph_tensor_acclelrator_for_general_gnn_b200 import build
    if shutil.which("cuobjdump") is None:
        pytest.skip("cuobjdump not on PATH")
    sass = subprocess.run(["cuobjdump", "-sass", build.build()], capture_output=True, text=True, check=True).stdout
    per_fn, fn = {}, None
    for line in sass.splitlines():
        if "Function :" in line:
            fn = line.split("Function :")[1].strip()
            per_fn[fn] = []
        elif fn is not None:
            per_fn[fn].append(line)
    assert "EF_CUDA_SM100" in sass or "sm_100" in sass
    has = lambda fn_part, mnemonic: any(fn_part in f and any(mnemonic in ln for ln in body) for f, body in per_fn.items())
    assert has("gemm_tc_kernel", "UTCHMMA"), "tcgen05.mma missing from gemm_tc_kernel"
    assert has("gemm_tc_kernel", "UTMALDG"), "TMA loads missing from gemm_tc_kernel"
    assert has("gemm_tc_kernel", "LDTM"), "tcgen05.ld (TMEM read-back) missing from gemm_tc_kernel"
    # mangled names (length-prefixed): "16aggregate_kernel" is the weighted aggregate only, not the GAT kernels
    for kernel in ("3gta20gat_aggregate_kernel", "3gta16aggregate_kernel", "3gta24gat_aggregate_llh_kernel"):
        assert has(kernel, "STRONG.SYS"), f"{kernel}: no system-scope access -- the exchange is not inside the launch"
    for kernel in ("3gta20gat_aggregate_kernel", "3gta16aggregate_kernel"):
        assert has(kernel, "LDGSTS"), f"{kernel}: cp.async staging of the next item is gone"
