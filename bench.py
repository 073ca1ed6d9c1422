#!/usr/bin/env python
"""Headline benchmark: GTEPS of one GAT layer on a Reddit-shape synthetic graph, executed from
the ISA program the reference's compiler.py -> interpreter.py emit (tests/golden/isa), on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dump-outputs DIR]

N > 1 is launched by torchrun (one rank per GPU); the graph is partitioned by destination range
(balanced by edges), each layer all-gathers Z and er over NCCL.  Prints ONE JSON line (rank 0).

A step = one full GAT layer (ops 0-13 of genGraphOP.py:49-62): GEMM X.W with the el/er
projections, single-pass edge softmax + aggregation + ELU.  ``value`` = E / step time with the
inputs resident in HBM; ``e2e`` = the same through ``execute()`` with HOST (pinned) features
copied in and the result copied out inside the timed region.

``--dump-outputs DIR`` writes the last timed step's layer output (``output.npy``) and the global row ids it
holds (``output_rows.npy``): every row, or a fixed seeded sample of rows beyond 64 MB.  With N > 1 only rank
0's destination rows are written; which rows rank 0 owns depends on N, so compare dumps taken with the same N.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

#: second layer of the two-layer workloads: (op graph, ISA program, output width)
SECOND_LAYER = {"flickr-gcn2": ("opgraph/GCN-flickr-layer2-trans.yaml", "isa/GCN-flickr-layer2-trans__0_1-2-3.yaml", 64)}

WORKLOADS = {
    # name: (shape, network, layer, reorder, opgraph yaml, isa yaml, heads)
    "reddit-gat": ("reddit", "GAT", 1, False, "opgraph/GAT-reddit-restamped-h4.yaml",
                   "isa/GAT-reddit-layer1-original__0-1-2_4-5-6-7-8_3-9-10-11-12-13.yaml", 4),
    "flickr-gat": ("flickr", "GAT", 1, False, "opgraph/GAT-flickr-layer1-original.yaml",
                   "isa/GAT-flickr-layer1-original__0-1-2_4-5-6-7-8_3-9-10-11-12-13.yaml", 16),
    "cora-gat": ("cora", "GAT", 1, False, "opgraph/GAT-cora-restamped-h4.yaml",
                 "isa/GAT-cora-layer1-original__0-1-2_4-5-6-7-8_3-9-10-11-12-13.yaml", 4),
    "flickr-gcn": ("flickr", "GCN", 1, True, "opgraph/GCN-flickr-layer1-trans.yaml",
                   "isa/GCN-flickr-layer1-trans__0_1-2-3.yaml", 0),
    "reddit-gcn": ("reddit", "GCN", 1, True, "opgraph/GCN-reddit-layer1-trans.yaml",
                   "isa/GCN-reddit-layer1-trans__0_1-2-3.yaml", 0),
    # BASELINE config 3: the 2-layer Flickr GCN (500 -> 128 -> 64), layer 1's (sharded) device output is layer 2's input
    "flickr-gcn2": ("flickr", "GCN", 1, True, "opgraph/GCN-flickr-layer1-trans.yaml",
                    "isa/GCN-flickr-layer1-trans__0_1-2-3.yaml", 0),
    # the Reddit shape with the heavier-tailed degree sequence (synthetic.HEAVY_TAIL: max degree 47x the mean)
    "reddit-heavy-gat": ("reddit-heavy", "GAT", 1, False, "opgraph/GAT-reddit-restamped-h4.yaml",
                         "isa/GAT-reddit-layer1-original__0-1-2_4-5-6-7-8_3-9-10-11-12-13.yaml", 4),
    "reddit-heavy-gcn": ("reddit-heavy", "GCN", 1, True, "opgraph/GCN-reddit-layer1-trans.yaml",
                         "isa/GCN-reddit-layer1-trans__0_1-2-3.yaml", 0),
}
F_OUT = 128


def resolve_workload(name):
    """WORKLOADS entry, or 'rmat<scale>-gcn': Graph500 RMAT graph (edge factor 16), 256 features, GCN layer
    (BASELINE config 5 at scale 24; the ISA program is the Reddit GCN-trans one, op sizes unchecked)."""
    import re
    m = re.fullmatch(r"rmat(\d+)-gcn", name)
    if m:
        return ("rmat%s" % m.group(1), "GCN", 1, True, "opgraph/GCN-reddit-layer1-trans.yaml",
                "isa/GCN-reddit-layer1-trans__0_1-2-3.yaml", 0)
    return WORKLOADS[name]


def shape_of(shape):
    from gta_graph_tensor_acclelrator_for_general_gnn_b200 import synthetic
    if shape.startswith("rmat"):
        scale = int(shape[4:])
        return (1 << scale), 16 << scale, 256
    return synthetic.SHAPES[shape[:-6] if shape.endswith("-heavy") else shape]


def f_out_of(shape):
    """Output width of the layer: 128 (genGraphOP.py:31-32 layer 1), 256 -> 256 for the RMAT config (BASELINE.md section 3)."""
    return 256 if shape.startswith("rmat") else F_OUT


def graph_of(shape):
    from gta_graph_tensor_acclelrator_for_general_gnn_b200 import synthetic
    if shape.startswith("rmat"):
        return synthetic.rmat_graph(int(shape[4:]))
    return synthetic.shape_graph(shape)


METRIC = "GTEPS per GAT/GCN layer (Reddit shape)"


def baseline_metric():
    """BASELINE.json's metric string, verbatim (``METRIC`` is its GTEPS half; the roofline object is the other)."""
    try:
        with open(os.path.join(REPO, "BASELINE.json")) as f:
            return json.load(f).get("metric")
    except (OSError, ValueError):
        return None


def load_yaml(rel):
    import yaml
    with open(os.path.join(REPO, "tests", "golden", rel)) as f:
        return yaml.safe_load(f)


def measured_peak():
    p = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def algorithmic_bytes(network, n, e, fin, f, h, s=4, sz=None):
    """SURVEY.md section 8d, no-reuse gather model.  Returns (layer bytes, dominant-kernel bytes).  ``sz`` = bytes per
    element of the gathered table Z (2 in the bf16 storage mode; X, el, er, edge weights and the output stay fp32)."""
    sz = s if sz is None else sz
    gemm = n * fin * s + fin * f * s + n * f * sz
    if network == "GAT":
        gemm += 2 * f * h * s + 2 * n * h * s
        edge = (n + 1) * 4 + e * 4 + e * h * s + n * h * s + e * f * sz + n * f * s
    else:
        edge = (n + 1) * 4 + e * (4 + s) + e * f * sz + n * f * s
    return gemm + edge, edge


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 50 ms during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, uuid):
        self.uuid, self.proc, self.lines = uuid, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", self.uuid, f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1]))
            except ValueError:
                continue
            for nm, val in zip(names, parts[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------
# CPU arm: the oracle's restatement on the host cores (the reference has no functional path)
# ------------------------------------------------------------------------------------------

def cpu_layer_sample(network, indptr_s, indices_s, row0, x, w, al, ar, edge_w_s):
    """One layer on the host: full GEMM (numpy BLAS, all threads) + the edge phase of the sample
    rows (C oracle, OpenMP).  Returns (t_gemm, t_edge) in seconds."""
    from oracle import c_oracle
    t0 = time.perf_counter()
    z = x @ w
    if network == "GAT":
        el = z @ al
        er = z @ ar
    t1 = time.perf_counter()
    rows = indptr_s.shape[0] - 1
    if network == "GAT":
        c_oracle.gat_edge_phase(indptr_s, indices_s, el[row0:row0 + rows], er, z, dtype=np.float32)
    else:
        c_oracle.spmm(indptr_s, indices_s, edge_w_s, z, dtype=np.float32)
    t2 = time.perf_counter()
    return t1 - t0, t2 - t1


def host_sample_csr(coo, n, sample_rows):
    """CSR of destination rows [0, sample_rows) of a host edge list (numpy)."""
    from oracle import gta_oracle as O
    keep = coo.dst < sample_rows
    d, s = coo.dst[keep], coo.src[keep]
    indptr, indices, _ = O.csr_build(d, s, sample_rows)
    return indptr, indices


def run_reference_arm(args, wl):
    """--impl reference: the CPU restatement of the path on this box's host cores, bounded sample."""
    from gta_graph_tensor_acclelrator_for_general_gnn_b200 import synthetic
    from oracle import c_oracle
    shape, network, layer, reorder, _, _, heads = wl
    note = ""
    if shape.startswith("rmat") and int(shape[4:]) > 20:
        # the host cannot hold the scale-24 inputs of this arm in bounded time: same generator at scale 20
        note = f" [sampled on RMAT-20 (same generator parameters, 1/{1 << (int(shape[4:]) - 20)} of the nodes and edges of {shape})]"
        shape = "rmat20"
    n, e, fin = shape_of(shape)
    coo = graph_of(shape)
    x, w, al, ar = synthetic.gat_tensors(n, fin, f_out_of(shape), max(heads, 1), seed=0)
    # sample = first rows holding about sample_edges edges
    deg = np.bincount(coo.dst, minlength=n)
    cum = np.cumsum(deg)
    sample_rows = int(min(n, max(64, np.searchsorted(cum, args.cpu_sample_edges) + 1)))
    indptr_s, indices_s = host_sample_csr(coo, n, sample_rows)
    e_s = int(indptr_s[-1])
    ew = None
    if network == "GCN":
        d = np.maximum(deg, 1).astype(np.float64)
        rows = np.repeat(np.arange(sample_rows), np.diff(indptr_s))
        ew = (1.0 / np.sqrt(d[rows] * d[indices_s])).astype(np.float32)
    c_oracle.use_all_cores()
    times = []
    for it in range(args.warmup + args.steps):
        tg, te = cpu_layer_sample(network, indptr_s, indices_s, 0, x, w, al, ar, ew)
        if it >= args.warmup:
            times.append((tg, te))
    tg = float(np.mean([t[0] for t in times]))
    te = float(np.mean([t[1] for t in times]))
    full = tg + te * e / max(e_s, 1)
    value = e / full / 1e9
    cores = os.cpu_count()
    sample = (f"full GEMM {n}x{fin}x{f_out_of(shape)} (numpy BLAS) + edge phase of dst rows [0,{sample_rows}) = {e_s} of {e} "
              f"edges (C oracle, OpenMP {c_oracle.threads()} threads); layer time extrapolated as "
              f"t_gemm + t_edge*E/E_sample" + note)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "GTEPS", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": (tg + te) * 1e3,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": {"workload": workload_name(args, wl), "baseline_metric": baseline_metric()},
            "cpu_baseline": {"value": value, "unit": "GTEPS", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": "GTEPS", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def workload_name(args, wl):
    shape, network, layer, reorder, _, isa_rel, heads = wl
    n, e, fin = shape_of(shape)
    h = f" H={args.heads or heads}" if network == "GAT" else ""
    if shape.startswith("rmat"):
        kind = "RMAT (a,b,c,d)=(0.57,0.19,0.19,0.05) edge factor 16, duplicates kept"
    elif shape.endswith("-heavy"):
        kind = "Chung-Lu P(rank)~(rank+600)^-0.9 (max degree ~47x mean, median ~0.41x)"
    else:
        kind = "Chung-Lu P(rank)~(rank+100)^-0.5 (max degree ~25x mean, median ~0.72x: milder than real Reddit, see DESIGN.md)"
    two = " + layer2 (128 -> 64) chained on the device" if args.workload in SECOND_LAYER else ""
    return (f"{network} layer{layer}{two} ({'trans' if reorder else 'original'}) on {shape}-shape synthetic graph "
            f"N={n} E={e} Fin={fin} F={f_out_of(shape)}{h} fp32, {kind}, program {os.path.basename(isa_rel)}")


def measured_traffic(workload, kernel, world):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel from an `ncu --set full` capture
    of THIS workload on one GPU (profiles/traffic.json names the capture); None when no capture exists for the shape
    being run (any N > 1: the per-rank launch has another shape)."""
    tp = os.path.join(REPO, "profiles", "traffic.json")
    if world != 1 or not os.path.exists(tp):
        return None, "no ncu capture of this launch shape"
    with open(tp) as f:
        entry = json.load(f).get(f"{workload}:{kernel}")
    if not entry:
        return None, "no ncu capture of this launch shape"
    return int(entry["bytes"]), entry["source"]


def reference_pipeline_timing(shape):
    """Wall-clock of the reference's own pipeline (compile -> interpret -> simulate, vTCAD/code/test.py:10-15) on the
    Cora-shape config, timed here on the box's host (one Python thread: the reference cannot use more).  Needs the
    reference files under baseline/_ref (git-ignored, copied by tools/install_reference.py); None when absent."""
    if shape != "cora":
        return None
    try:
        sys.path.insert(0, os.path.join(REPO, "tools"))
        import reference_pipeline
        return reference_pipeline.time_pipeline(os.path.join(REPO, "baseline", "_ref"))
    except Exception as exc:      # a reported baseline, never a requirement
        return {"unavailable": str(exc).splitlines()[0][:160] if str(exc) else type(exc).__name__}


def parity_big(P, torch, y_h, ip_s, ix_s, rows_sel, edge_w_rows, x_d, w_d, z_local, table, part):
    """Parity for shapes whose whole-output oracle does not fit the host (RMAT-24): (1) the aggregation of the sampled
    rows against the fp64 oracle applied to the SOURCE ROWS THE KERNEL GATHERED (fetched from the device table), (2) the
    GEMM on sampled rows against fp64 X.W.  Both under the stated tolerance; the worse of the two is reported."""
    uniq, inv = np.unique(ix_s, return_inverse=True)
    if part is not None:
        b = np.asarray(part.bounds, dtype=np.int64)
        owner = np.searchsorted(b, uniq, side="right") - 1
        slot = (owner - part.rank) % part.world if part.rotate else owner
        table_rows = slot * part.stride + (uniq - b[owner])
    else:
        table_rows = uniq
    z_rows = table[torch.from_numpy(table_rows).to(table.device)].cpu().numpy().astype(np.float64)
    rep = P.check_gcn(y_h, ip_s, inv.astype(np.int32), edge_w_rows, z_rows, np.abs(z_rows))
    # GEMM rows
    k = min(4096, int(z_local.shape[0]))
    pick = torch.linspace(0, z_local.shape[0] - 1, k, device=z_local.device).long()
    x64 = x_d[pick].cpu().numpy().astype(np.float64)
    w64 = w_d.cpu().numpy().astype(np.float64)
    z64 = x64 @ w64
    zs = np.abs(x64) @ np.abs(w64)
    zerr = np.abs(z_local[pick].cpu().numpy().astype(np.float64) - z64) / (P.RTOL * np.abs(z64) + P.RTOL * zs + 1e-30)
    rep["gemm_rows_checked"] = k
    rep["gemm_max_err_over_tol"] = float(zerr.max())
    rep["aggregate_max_err_over_tol"] = rep["max_err_over_tol"]
    rep["max_err_over_tol"] = max(rep["max_err_over_tol"], float(zerr.max()))
    rep["mode"] = ("aggregation of the sampled rows vs fp64 oracle on the source rows fetched from the device table + GEMM "
                   "on %d sampled rows vs fp64 X.W (whole-output oracle does not fit the host at this shape)" % k)
    return rep


DUMP_BYTES = 64 * 10**6 - 4096      # --dump-outputs budget, .npy headers included


def dump_outputs(out_dir, y, row0):
    """--dump-outputs: ``y`` (rank 0's output rows, global ids from ``row0``; every row when N = 1) as float32, every
    row when it fits DUMP_BYTES, else the same seeded sample of rows on every run of the same shape."""
    rows, cols = int(y.shape[0]), int(y.shape[1])
    keep = min(rows, DUMP_BYTES // (cols * 4 + 8))
    pick = np.arange(rows) if keep == rows else np.sort(np.random.default_rng(0).choice(rows, keep, replace=False))
    import torch
    vals = y[torch.from_numpy(pick).to(y.device)].float().cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "output.npy"), vals)
    np.save(os.path.join(out_dir, "output_rows.npy"), (pick + row0).astype(np.float64))


# ------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------

def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="reddit-gat", help="one of %s or rmat<scale>-gcn" % sorted(WORKLOADS))
    ap.add_argument("--heads", type=int, default=0, help="override the attention width H")
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--cpu-sample-edges", type=int, default=40_000_000,
                    help="edges in the CPU arm's sample (whole destination rows from row 0); the layer time is "
                         "extrapolated from it.  40 M edges = about a second per step on 16 cores")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the fp64-oracle check of the benchmarked output")
    ap.add_argument("--parity-edges", type=int, default=200_000_000,
                    help="edge budget of the parity check: every destination row of rank 0 when it holds at most this "
                         "many edges, else the 512 highest-degree rows plus every k-th row")
    ap.add_argument("--no-fuse", action="store_true", help="honour every STORE_* of the program")
    ap.add_argument("--exchange", default="fused", choices=["fused", "nccl"],
                    help="multi-GPU source exchange: pulled over NVLink inside the aggregation launch (default), or one "
                         "NCCL all-gather per layer (the round-1 path, kept as the baseline)")
    ap.add_argument("--copy-ctas", type=int, default=0, help="fused exchange: CTAs that pull (0 = library default)")
    ap.add_argument("--no-graph", action="store_true", help="issue kernels eagerly instead of replaying a CUDA graph")
    ap.add_argument("--dtype", default="f32", choices=["f32", "bf16"],
                    help="bf16 = bf16 STORAGE MODE: the gathered table Z in bf16, fp32 accumulation (its own tolerance: "
                         "rtol 2e-2, atol 1e-2 rowscale); never the headline")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the layer output of the last timed step to DIR/output.npy (float32; rank 0's rows) and "
                         "the global row ids it holds to DIR/output_rows.npy (float64): every row when both fit "
                         "64 MB, else a fixed seeded sample of rows, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    wl = resolve_workload(args.workload)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes the GPU path's output; --impl reference times a host sample")
        if rank == 0:
            run_reference_arm(args, wl)
        return

    import torch
    import torch.distributed as dist
    from gta_graph_tensor_acclelrator_for_general_gnn_b200 import _cabi, executor, graph, isa, kernels, synthetic
    from gta_graph_tensor_acclelrator_for_general_gnn_b200 import dist as gdist

    lib = _cabi.load()      # no CUDA extension => fail here, loudly
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a GPU (there is no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    shape, network, layer, reorder, op_rel, isa_rel, heads = wl
    heads = args.heads or heads
    n, e, fin = shape_of(shape)
    f_out = f_out_of(shape)
    big = shape.startswith("rmat") and n > (1 << 21)      # too big for host-side inputs and a whole-output oracle
    op_info = load_yaml(op_rel)
    program = isa.Program.from_records(load_yaml(isa_rel))
    second = SECOND_LAYER.get(args.workload)
    if second is not None:
        op_info2, program2, f_out2 = load_yaml(second[0]), isa.Program.from_records(load_yaml(second[1])), second[2]

    # ---- inputs (synthetic, deterministic) ---------------------------------------------------
    t_setup = time.perf_counter()
    if shape.startswith("rmat"):
        dst_d, src_d, _ = synthetic.rmat_graph_device(int(shape[4:]), device=dev)
        graph_checksum = "device-generated RMAT, seed 0: sum(dst)=%d sum(src)=%d" % (int(dst_d.sum(dtype=torch.int64)),
                                                                                     int(src_d.sum(dtype=torch.int64)))
        degree_stats = None
    else:
        coo = graph_of(shape)
        graph_checksum = coo.checksum()
        degree_stats = synthetic.degree_stats(coo.dst, n) if rank == 0 else None
        dst_d, src_d = torch.from_numpy(coo.dst).to(dev), torch.from_numpy(coo.src).to(dev)
        del coo
    deg_d = torch.bincount(dst_d, minlength=n)          # global in-degrees (GCN edge norm)
    if world > 1:
        part = gdist.partition_from_coo(dst_d, src_d, n, rank, world, rotate=(args.exchange == "fused"))
        g, r0, r1 = part.local, part.row_begin, part.row_end
        exchange = gdist.FusedExchange(part, copy_ctas=args.copy_ctas) if args.exchange == "fused" else gdist.SourceExchange(part)
        # global source id of every local edge (the remap inverted): slot -> owner, offset inside the owner's rows
        slot = torch.div(g.indices, part.stride, rounding_mode="floor")
        owner = (slot + (rank if part.rotate else 0)) % world
        bounds_t = torch.tensor(part.bounds, dtype=torch.int64, device=dev)
        src_glob = bounds_t[owner.long()] + (g.indices - slot * part.stride).long()
        del slot, owner
    else:
        part = None
        g = graph.csr_from_coo(dst_d, src_d, n)
        r0, r1, exchange = 0, n, None
        src_glob = g.indices.long()
    del dst_d, src_d
    torch.cuda.empty_cache()
    e_local = g.num_edges
    edge_w = None
    if network == "GCN":      # 1/sqrt(deg_i deg_j) in the local graph's edge order
        deg = deg_d.clamp(min=1).to(torch.float64)
        rows_of_edge = torch.repeat_interleave(torch.arange(r0, r1, device=dev), g.indptr[1:] - g.indptr[:-1])
        edge_w = (1.0 / torch.sqrt(deg[rows_of_edge] * deg[src_glob])).to(torch.float32)[:, None].contiguous()
        del rows_of_edge, deg
    parity_csr = None
    if rank == 0 and not args.no_parity:      # rank 0's rows with GLOBAL source ids, on the host
        parity_csr = (g.indptr.cpu().numpy(), src_glob.to(torch.int32).cpu().numpy())
    host_csr = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline and not big:      # the CPU leg is an N = 1 item
        ip_h = g.indptr.cpu().numpy()
        deg_h = np.diff(ip_h)
        sample_rows = int(min(n, max(64, np.searchsorted(np.cumsum(deg_h), args.cpu_sample_edges) + 1)))
        e_s = int(ip_h[sample_rows])
        host_csr = (ip_h[:sample_rows + 1].copy(), g.indices[:e_s].cpu().numpy(), sample_rows, deg_h)
    del src_glob
    torch.cuda.empty_cache()
    if big:      # features and weights drawn on the device: rank p's rows from generator seed 1000 + p
        gen = torch.Generator(device=dev).manual_seed(1000 + rank)
        x_d = kernels.alloc_table(r1 - r0, fin, dev)
        x_d.normal_(generator=gen)
        gen_w = torch.Generator(device=dev).manual_seed(7)
        lim = float(np.sqrt(6.0 / (fin + f_out)))
        w_d = (torch.rand((fin, f_out), device=dev, generator=gen_w) * 2 - 1) * lim
        x_h = w_h = al_h = ar_h = None
        x_pin = None
        weights = {0: w_d}
    else:
        x_h, w_h, al_h, ar_h = synthetic.gat_tensors(n, fin, f_out, max(heads, 1), seed=0)
        x_pin = torch.from_numpy(x_h[r0:r1]).pin_memory()
        x_d = kernels.to_table(x_pin.to(dev))
        w_d, al_d, ar_d = (torch.from_numpy(a).to(dev) for a in (w_h, al_h, ar_h))
        weights = {0: w_d, 1: al_d, 2: ar_d} if network == "GAT" else {0: w_d}
    final_op = len(op_info) - 1
    edge_inputs = {2: edge_w} if network == "GCN" else None
    if second is not None:
        w2_h = synthetic.glorot(np.random.default_rng(11), f_out, f_out2)
        weights2 = {0: torch.from_numpy(w2_h).to(dev)}
    torch.cuda.synchronize()
    t_setup = time.perf_counter() - t_setup

    feature_dtype = torch.bfloat16 if args.dtype == "bf16" else torch.float32
    sz = 2 if args.dtype == "bf16" else 4

    def step(x_dev):
        y1 = executor.execute(program, op_info, g, {0: x_dev}, weights, edge_inputs, network=network,
                              is_reorder=reorder, fuse_across_blocks=not args.no_fuse, source_table=exchange,
                              check_shapes=(world == 1 and not shape.startswith("rmat")),
                              feature_dtype=feature_dtype)[final_op]
        if second is None:
            return y1
        # layer 2 on layer 1's output: the rows this rank owns are the rows it just computed -- no host round trip,
        # no re-partition; only the layer's own source exchange moves data between the GPUs
        return executor.execute(program2, op_info2, g, {0: y1}, weights2, edge_inputs, network=network,
                                is_reorder=reorder, fuse_across_blocks=not args.no_fuse, source_table=exchange,
                                check_shapes=(world == 1), feature_dtype=feature_dtype)[len(op_info2) - 1]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        y = step(x_d)
    barrier()

    # the timed step: the same execute() call, captured once into a CUDA graph and replayed
    graphed = None
    graph_note = "eager"
    if world > 1:
        # the fused exchange carries a step number and alternates two tables; steps are issued eagerly
        # (host enqueue time is reported; it hides under the previous step's kernels)
        graph_note = "eager (multi-rank: per-step exchange state lives on the host)"
    elif not args.no_graph:
        try:
            graphed = executor.GraphedExecution(lambda: step(x_d))
            graph_note = "cuda graph replay of execute()"
        except Exception as exc:      # capture is an optimisation, never a requirement
            graphed = None
            graph_note = "eager (graph capture failed: %s)" % str(exc).splitlines()[0][:120]
            torch.cuda.synchronize()
    run_step = (lambda: graphed.replay()) if graphed is not None else (lambda: step(x_d))
    for _ in range(args.warmup):
        y = run_step()
    barrier()

    # ---- timed region: K steps, resident inputs ---------------------------------------------
    props = torch.cuda.get_device_properties(dev)
    sampler = ClockSampler("GPU-" + str(props.uuid) if hasattr(props, "uuid") else str(local_rank))
    if rank == 0:
        sampler.start()
    lib.gta_launch_count_reset()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    host_t0 = time.perf_counter()
    for _ in range(args.steps):
        y = run_step()
    host_ms = (time.perf_counter() - host_t0) * 1e3 / args.steps      # CPU time to ENQUEUE a step
    ev1.record()
    barrier()
    elapsed_ms = ev0.elapsed_time(ev1)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:      # before more steps run: a replayed graph reuses its output buffer
        dump_outputs(args.dump_outputs, y, r0)
    t = torch.tensor([elapsed_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_per_step = float(t.item()) / args.steps
    layers = 2 if second is not None else 1
    value = layers * e / (ms_per_step * 1e-3) / 1e9          # GTEPS per layer: every layer walks all E edges

    # per-kernel durations: the same K steps issued eagerly with CUDA events around every kernel.  One untimed eager
    # step first: the timed region above replayed a CUDA graph, so this is the first eager launch on this stream and
    # it allocates that stream's chain-state workspace (1 GB on RMAT-20) inside what would be the first interval
    y = step(x_d)
    kernels.EVENT_LOG = []
    lib.gta_launch_count_reset()
    barrier()
    for _ in range(args.steps):
        y = step(x_d)
    barrier()
    launches = int(lib.gta_launch_count())
    log, kernels.EVENT_LOG = kernels.EVENT_LOG, None
    per_kernel = {}
    for name, a, b in log:
        per_kernel.setdefault(name, []).append(a.elapsed_time(b))

    # ---- e2e: host features in, result out, through execute() -------------------------------
    # Every step copies ITS features from pinned host memory and ITS result back; the copies of
    # neighbouring steps overlap this step's kernels (pipeline.HostPipeline: 3 streams, 2 buffers).
    e2e = None
    if not args.no_e2e and x_pin is not None:
        from gta_graph_tensor_acclelrator_for_general_gnn_b200 import pipeline
        xs_pin = []
        for _ in range(2):
            t_pin = pipeline.pinned_table(r1 - r0, fin)
            t_pin.copy_(x_pin)
            xs_pin.append(t_pin)
        ys_pin = [torch.empty((r1 - r0, f_out2 if second is not None else f_out), dtype=torch.float32).pin_memory()
                  for _ in range(2)]

        def e2e_run(pipe, steps):
            barrier()
            for i in range(steps):
                pipe.submit(xs_pin[i % 2], ys_pin[i % 2])
            ms = pipe.finish()
            barrier()
            tt = torch.tensor([ms], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            return float(tt.item()) / steps

        # one pipeline object per mode, warmed first: the caching allocator keeps per-stream pools, so the
        # first steps on fresh streams pay cudaMalloc (device-synchronising) for Z / el / er / out
        pipe2 = pipeline.HostPipeline(step, r1 - r0, fin, dev, depth=2)
        pipe1 = pipeline.HostPipeline(step, r1 - r0, fin, dev, depth=1)
        e2e_run(pipe2, 5)
        e2e_run(pipe1, 3)
        e2e_serial_ms = e2e_run(pipe1, max(args.e2e_steps // 2, 2))
        e2e_ms = e2e_run(pipe2, args.e2e_steps)
        assert torch.equal(ys_pin[0], y.cpu()), "e2e result differs from the resident-input result"
        h2d = int(xs_pin[0].numel() * 4)
        d2h = int(ys_pin[0].numel() * 4)
        # the ceiling of this box: every rank uploads its features at the same time, nothing else running
        stage = pipe2.stage[0]
        flat_src = torch.as_strided(xs_pin[0], (xs_pin[0].shape[0] * xs_pin[0].stride(0),), (1,))
        flat_dst = torch.as_strided(stage, (stage.shape[0] * stage.stride(0),), (1,))
        barrier()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record()
        for _ in range(3):
            flat_dst.copy_(flat_src, non_blocking=True)
        c1.record()
        barrier()
        tc = torch.tensor([c0.elapsed_time(c1) / 3], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tc, op=dist.ReduceOp.MAX)
        h2d_ms = float(tc.item())
        e2e = {"value": layers * e / (e2e_ms * 1e-3) / 1e9, "unit": "GTEPS", "ms_per_step": e2e_ms,
               "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "serial_ms_per_step": e2e_serial_ms,
               "h2d_alone_ms": h2d_ms, "h2d_alone_gbs_per_rank": h2d / (h2d_ms * 1e-3) / 1e9,
               "note": "per rank and per step: features X (pinned host) -> device, execute(), result -> pinned "
                       "host, all inside the timed region; copies of neighbouring steps overlap the kernels "
                       "(pipeline.HostPipeline, depth 2; serial_ms_per_step = depth 1); the CSR (static graph "
                       "structure) and the weights stay resident.  h2d_alone_ms = the same upload on every rank at "
                       "once with nothing else running (max over ranks): the host-side floor of a step"}

    # bitwise run-to-run reproducibility of the timed path (every rank; the reduction shape is fixed)
    y_first = run_step().clone()
    bitwise = bool(torch.equal(y_first, run_step()))
    if world > 1:
        tb = torch.tensor([int(bitwise)], dtype=torch.int32, device=dev)
        dist.all_reduce(tb, op=dist.ReduceOp.MIN)
        bitwise = bool(tb.item())
    barrier()
    z_dev = big_table = None
    if big and not args.no_parity:
        # one more step (every rank, so the exchange stays in step) that also returns Z, and the table it gathered from
        z_dev = executor.execute(program, op_info, g, {0: x_d}, weights, edge_inputs, network=network, is_reorder=reorder,
                                 source_table=exchange, check_shapes=False, outputs=[0, final_op])
        torch.cuda.synchronize()
        big_table = exchange.last_table(f_out) if exchange is not None else z_dev[0]
    barrier()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- parity of the BENCHMARKED output against the fp64 oracle (rank 0's destination rows) ----------
    parity = None
    if parity_csr is not None:
        from oracle import c_oracle, parity as P
        c_oracle.use_all_cores()
        t_par = time.perf_counter()
        indptr_l, indices_l = parity_csr
        budget = min(args.parity_edges, 4_000_000) if big else args.parity_edges
        rows_sel = P.select_rows(indptr_l, budget)
        ip_s, ix_s = P.sub_csr(indptr_l, indices_l, rows_sel)
        y_h = y_first.cpu().numpy()[rows_sel]
        tol = P.BF16 if args.dtype == "bf16" else P.RTOL
        if big:
            deg_l = np.diff(indptr_l)
            pos = np.repeat(indptr_l[rows_sel] - ip_s[:-1], deg_l[rows_sel]) + np.arange(int(ip_s[-1]), dtype=np.int64)
            ew_rows = edge_w.reshape(-1)[torch.from_numpy(pos).to(dev)].cpu().numpy()
            parity = parity_big(P, torch, y_h, ip_s, ix_s, rows_sel, ew_rows, x_d, w_d, z_dev[0], big_table, part)
        elif network == "GAT":
            z64, zabs, el64, er64 = P.host_tables(x_h, w_h, al_h, ar_h)
            parity = P.check_gat(y_h, ip_s, ix_s, el64[r0 + rows_sel], er64, z64, zabs, rtol=tol)
        else:
            z64, zabs, _, _ = P.host_tables(x_h, w_h)
            deg_l = np.diff(indptr_l)
            pos = np.repeat(indptr_l[rows_sel] - ip_s[:-1], deg_l[rows_sel]) + np.arange(int(ip_s[-1]), dtype=np.int64)
            ew_rows = edge_w.cpu().numpy().reshape(-1)[pos]
            if second is not None:
                # whole chain in fp64: layer 1 over the WHOLE graph (layer 2 gathers from every node), its error scale
                # carried into layer 2 (3 x: layer 1's output error <= 2e-5 scale, plus layer 2's own product)
                from oracle import gta_oracle as O
                coo_h = graph_of(shape)
                ip_f, ix_f, _ = O.csr_build(coo_h.dst, coo_h.src, n)
                ew_f = synthetic.gcn_edge_norm(ip_f, ix_f).astype(np.float64)
                y1 = c_oracle.spmm(ip_f, ix_f, ew_f, z64, dtype=np.float64)
                s1 = c_oracle.spmm(ip_f, ix_f, ew_f, zabs, dtype=np.float64)
                z64, zabs = y1 @ w2_h.astype(np.float64), 3.0 * s1 @ np.abs(w2_h).astype(np.float64)
            parity = P.check_gcn(y_h, ip_s, ix_s, ew_rows, z64, zabs, rtol=tol)
        parity.update(bitwise_rerun=bitwise, rows_of=int(r1 - r0), edges_of=int(indptr_l[-1]),
                      checked="rank 0's destination rows [%d,%d)%s" % (r0, r1, "" if rows_sel.shape[0] == r1 - r0 else
                                                                      " (512 highest-degree rows + every k-th row)"),
                      seconds=round(time.perf_counter() - t_par, 1))

    # ---- roofline of the dominant kernel ------------------------------------------------------
    dom = "gta_gat_aggregate_f32" if network == "GAT" else "gta_aggregate_f32"
    dom_ms = float(np.mean(per_kernel[dom][0::layers])) if dom in per_kernel else None      # (layer 1's launch)
    _, dom_bytes = algorithmic_bytes(network, r1 - r0, e_local, fin, f_out, max(heads, 1), sz=sz)
    layer_bytes, _ = algorithmic_bytes(network, n, e, fin, f_out, max(heads, 1), sz=sz)
    if second is not None:
        layer_bytes += algorithmic_bytes(network, n, e, f_out, f_out2, 1, sz=sz)[0]
    peak, peak_src = measured_peak()
    traffic, traffic_src = measured_traffic(args.workload, dom, world)
    roofline = None
    if dom_ms:
        ach = dom_bytes / (dom_ms * 1e-3) / 1e9
        # the gather term alone against the MEASURED gather ceiling of this device (L2-resident random rows, the
        # kernel's own load instruction): what the kernel is actually bound by when the table (or its column block)
        # fits L2.  Not meaningful when the table is far larger than L2 (RMAT-24: HBM-bound, use frac).
        gp = kernels.gather_peak(f=min(f_out * sz // 4, 128))      # same row BYTES as the kernel gathers
        gather_bytes = e_local * f_out * sz
        roofline = {"bound": "hbm", "kernel": dom, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                    "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                    "algorithmic_bytes_per_launch": dom_bytes, "kernel_ms": dom_ms,
                    "l2_gather_peak_gbs": gp["gbs"], "l2_gather_peak_how": "%s, %d-byte rows of a %.0f MB table" % (
                        gp["how"], gp["row_bytes"], gp["table_mb"]),
                    "l2_frac": gather_bytes / (dom_ms * 1e-3) / 1e9 / gp["gbs"],
                    "layer_frac": layer_bytes / (ms_per_step * 1e-3) / 1e9 / peak / max(world, 1),
                    "kernel_ms_by_name": {k: float(np.mean(v)) for k, v in per_kernel.items()},
                    "note": "frac = algorithmic bytes (no-reuse gather model, SURVEY 8d) / kernel time / measured HBM peak: "
                            "above 1 because L2 serves the re-reads; l2_frac = gathered row bytes / kernel time / measured "
                            "L2 gather peak is the fraction of the unit that actually bounds the kernel"}

    cpu_baseline = None
    if host_csr is not None:
        indptr_s, indices_s, sample_rows, deg_h = host_csr
        ew_s = None
        if network == "GCN":
            d = np.maximum(deg_h, 1).astype(np.float64)
            rows = np.repeat(np.arange(sample_rows), np.diff(indptr_s))
            ew_s = (1.0 / np.sqrt(d[rows] * d[indices_s])).astype(np.float32)
        from oracle import c_oracle
        c_oracle.use_all_cores()
        cpu_layer_sample(network, indptr_s[:65], indices_s[:int(indptr_s[64])], 0, x_h, w_h, al_h, ar_h, ew_s)  # warm
        # repeat the sample until about 10 s of CPU work have been timed (at most 40 passes), report the mean
        reps, t_begin = [], time.perf_counter()
        while len(reps) < 40 and (not reps or time.perf_counter() - t_begin < 10.0):
            reps.append(cpu_layer_sample(network, indptr_s, indices_s, 0, x_h, w_h, al_h, ar_h, ew_s))
        tg = float(np.mean([r[0] for r in reps]))
        te = float(np.mean([r[1] for r in reps]))
        e_s = int(indptr_s[-1])
        full_t = tg + te * e / max(e_s, 1)
        cpu_baseline = {"value": e / full_t / 1e9, "unit": "GTEPS", "cores": os.cpu_count(), "kind": "port",
                        "threads": c_oracle.threads(),
                        "sample": (f"full GEMM (numpy BLAS, {tg:.2f} s) + edge phase of dst rows [0,{sample_rows}) = "
                                   f"{e_s} of {e} edges (C oracle fp32, {te:.2f} s); mean of {len(reps)} passes; layer "
                                   f"time extrapolated as t_gemm + t_edge*E/E_sample")}
        ref_pipe = reference_pipeline_timing(shape)
        if ref_pipe is not None:
            cpu_baseline["reference_pipeline"] = ref_pipe

    if world > 1:
        par = f"dst-range partition x{world} (partition on build), " + (
            "[Z|er] pulled from the peers over NVLink inside the aggregation launch (no NCCL in the step)"
            if args.exchange == "fused" else "one NCCL all-gather of [Z|er] per layer")
    else:
        par = "single GPU"
    line = {"metric": METRIC, "value": value, "unit": "GTEPS", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
            "config": {"workload": workload_name(args, wl) + (" [bf16 storage of Z, fp32 accumulate]" if args.dtype == "bf16" else ""),
                       "baseline_metric": baseline_metric(), "parallelism": par,
                       "degrees": degree_stats,
                       "l2": "inputs larger than L2: CSR indices %.0f MB + X %.0f MB + Z %.0f MB re-read every step" % (
                           e * 4 / 1e6, n * fin * 4 / 1e6, n * f_out * 4 / 1e6),
                       "fuse_across_blocks": not args.no_fuse, "launch": graph_note,
                       "host_enqueue_ms_per_step": round(host_ms, 3), "graph_checksum": graph_checksum,
                       "setup_s": round(t_setup, 1)},
            "clocks": clocks, "e2e": e2e, "gpu_launches": launches,
            "roofline": roofline, "cpu_baseline": cpu_baseline, "parity": parity}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    if parity is not None and not (parity["max_err_over_tol"] <= 1.0 and parity["bitwise_rerun"]):
        raise SystemExit("parity FAILED: the benchmarked output is %.2fx the tolerance away from the fp64 oracle "
                         "(bitwise rerun: %s)" % (parity["max_err_over_tol"], parity["bitwise_rerun"]))


if __name__ == "__main__":
    main()
