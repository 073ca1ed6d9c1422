"""Partitioned layers on real ranks: one process and one GPU per rank, NCCL default group, data that changes every step.

The other exchange tests emulate every rank in one process on one GPU, where each step runs every rank's producer before
any consumer and every "peer" table sits in the same L2.  Here the ranks are processes on their own GPUs, so what only a
real run exercises runs too: the CUDA IPC mapping (gta_ipc_export / gta_ipc_open), the release store of `ready` seen by
a copy CTA on another GPU, copy CTAs that wait on a peer that has not published yet, ranks that run a step ahead of a
slow peer (the double-buffered tables and stats[step & 1] are safe only by the ordering argument in dist.py), ranks
without rows that launch no aggregation at all, the NCCL all-gather of dist.SourceExchange and the whole-table
all-gather plus roll of FusedExchange.__call__ (PNA's edge sum).

Every world size runs all its cases in one mp.spawn.  Each case runs 4 steps on data d0 d1 d2 d0, enqueued without a host
synchronise between them; at steps 2 and 3 one rank delays its step on the device and another on the host (at most
about 40 ms: the waits of the exchange trap only after 2^27 polls).  The workers write every rank's outputs; the tests
below check them in the parent against the fp64 oracle, step 4 against step 1, the single-process emulation of the same
partition (bit for bit: real peers change where the bytes come from, not the reduction order) and, for the NCCL
all-gather layout, the single-GPU run (bit for bit where the reduction order is the same).
"""
import os
import socket
import time
import traceback

import numpy as np
import pytest
import yaml

from conftest import assert_close_rowscale
from oracle import gta_oracle as O
from gta_graph_tensor_acclelrator_for_general_gnn_b200 import _cabi, synthetic
from test_gpu_bf16 import _assert_bf16_close
from test_gpu_exchange import (_aggregate_step, _er_max_per_owner, _gat_data, _gat_step, _host_graph, _hub_graph,
                               _inputs, _owner_of_rows, _stale_bound_breaks, assert_slots_hold, emulated, release)
from test_gpu_instances import crafted_graph
from test_gpu_kernels import _gat_from_z

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
WORLDS = (2, 5, 8)
STEPS = (0, 1, 2, 0)
#: device delay of the slow rank at steps 2 and 3 (SM clock cycles: 15 ms at 1965 MHz, below 40 ms above 750 MHz)
SLEEP_CYCLES = 30_000_000
HOST_DELAY_S = 0.02

#: kernel-level cases: (kind, dtype, f, heads); GCN aggregates 64 features with permuted edge weights
KERNEL_CALLS = {"gat-f32-h4": ("gat", "f32", 128, 4), "gat-f32-h3": ("gat", "f32", 96, 3),
                "gat-f32-h32": ("gat", "f32", 128, 32), "gat-bf16-h4": ("gat", "bf16", 128, 4),
                "gcn": ("gcn", "f32", 64, 0)}
GAT_ISA = "GAT-cora-layer1-original__0-1-2_4-5-6-7-8_3-9-10-11-12-13"
#: execute() cases: (ISA program, op graph, network, reorder, exchange, feature dtype); the bf16 GAT runs the 4-head op
#: graph of the same program (the bf16 single-pass kernel takes 1, 2 or 4 heads)
EXEC_CASES = {
    f"{net}-{ex}": (isa, opg, net, reorder, ex, "f32")
    for net, isa, opg, reorder in (
        ("GAT", GAT_ISA, "GAT-cora-layer1-original", False),
        ("GCN", "GCN-cora-layer1-trans__0_1-2-3", "GCN-cora-layer1-trans", True),
        ("DGN", "DGN-cora-layer2-original__0-1-2-3-4-5-6-7-8-9-10", "DGN-cora-layer2-original", False),
        ("PNA", "PNA-cora-layer2-original__0-1-2-3-4-5-6-7-8-9-10", "PNA-cora-layer2-original", False))
    for ex in ("fused", "nccl")}
EXEC_CASES["GAT-fused-bf16"] = (GAT_ISA, "GAT-cora-restamped-h4", "GAT", False, "fused", "bf16")


def _graphs(world):
    return ("crafted", "hub") if world == 8 else ("crafted",)


def _kernel_cases(world):
    return [f"{g}-{c}-copy{cc}" for g in _graphs(world) for c in KERNEL_CALLS for cc in (0, 1)]


def _exec_cases(world):
    return list(EXEC_CASES)


def _graph_coo(name):
    return crafted_graph() if name == "crafted" else _hub_graph()


def _load(rel):
    with open(os.path.join(GOLDEN, rel)) as fh:
        return yaml.safe_load(fh)


def _exec_inputs(op_info, n, e, d):
    """Weights of seed 0 at every step; node and edge inputs of data set d."""
    _, weights, _ = synthetic.opgraph_inputs(op_info, n, e, 0)
    node_inputs, _, edge_inputs = synthetic.opgraph_inputs(op_info, n, e, 100 + d)
    return node_inputs, weights, edge_inputs


# ---- the worker: one process per rank ---------------------------------------------------------------------------------
def _skew(s, rank, world):
    """At steps 2 and 3 rank s mod W starts late on the device, rank (s + 1) mod W on the host."""
    import torch
    if s in (1, 2):
        if rank == s % world:
            torch.cuda._sleep(SLEEP_CYCLES)
        elif rank == (s + 1) % world:
            time.sleep(HOST_DELAY_S)


def _agreed(setup, group, world):
    """Run ``setup()`` on every rank, then agree over gloo that it succeeded everywhere before any rank enqueues an
    aggregation that would wait for a peer's publish: a rank that failed raises, and so does every other rank."""
    import torch.distributed as dist
    ok, err, value = True, "", None
    try:
        value = setup()
    except Exception:
        ok, err = False, traceback.format_exc()
    agreed = [None] * world
    dist.all_gather_object(agreed, (ok, err), group=group)
    bad = [a[1] for a in agreed if not a[0]]
    if bad:
        raise RuntimeError("set-up failed on a rank:\n" + bad[0])
    return value


def _partition(host, n, rank, world, rotate):
    """bench.py's partition on build, fed the edge list in global CSR order: the rank's edges then arrive in the global
    CSR order of its rows, which is what ``Partition.permute_edges`` maps from."""
    import torch
    from gta_graph_tensor_acclelrator_for_general_gnn_b200 import dist as gdist
    dst = torch.from_numpy(O.row_ids(host.indptr).astype(np.int32)).cuda()
    src = torch.from_numpy(host.indices.astype(np.int32)).cuda()
    return gdist.partition_from_coo(dst, src, n, rank, world, rotate=rotate)


def _kernel_case(case, rank, world, coo, host, gloo):
    """Four steps of one kernel-level case through a real FusedExchange.  Returns {name: array}."""
    import torch
    from gta_graph_tensor_acclelrator_for_general_gnn_b200 import dist as gdist, kernels
    name = case.split("-copy")[0].split("-", 1)[1]
    call, copy_ctas = KERNEL_CALLS[name], int(case.rsplit("copy", 1)[1])
    n = coo[0]

    def setup():
        p = _partition(host, n, rank, world, True)
        return p, gdist.FusedExchange(p, copy_ctas=copy_ctas)
    part, ex = _agreed(setup, gloo, world)
    owner = _owner_of_rows(part.bounds, n)
    r0, r1 = part.row_begin, part.row_end
    e0, e1 = int(host.indptr[r0]), int(host.indptr[r1])
    ew = torch.from_numpy(synthetic.gcn_edge_norm(host.indptr, host.indices)).cuda()
    data = {}          # every data set on the device before the first step: no host copy between steps
    for d in set(STEPS):
        if call[0] == "gat":
            z, el, er = _gat_data(call, d, owner)
            zd = torch.from_numpy(z).cuda()
            zd = zd.to(torch.bfloat16) if call[1] == "bf16" else zd
            data[d] = (zd, torch.from_numpy(er).cuda(), torch.from_numpy(np.ascontiguousarray(el[r0:r1])).cuda())
        else:
            data[d] = (torch.from_numpy(_inputs(("gcn", "multiprocess"), f"x{d}", (n, 64))).cuda(),)
    torch.cuda.synchronize()
    steps = []
    for s, d in enumerate(STEPS):
        if call[0] == "gat":
            zd, erd, eld = data[d]
            wants = (zd, erd)
        else:
            zd, = data[d]
            wants = (zd,)
        _skew(s, rank, world)
        if call[0] == "gat":
            zt, ert, gate = ex.gather_pair(zd[r0:r1], erd[r0:r1])
            bounded = kernels.gat_aggregate(part.local, eld, ert, zt, exchange=gate)
            online = kernels.gat_aggregate(part.local, eld, ert, zt, exchange=gate, want_stats=True)
            outs = {"bounded": bounded.clone(), "online": online[0].clone(), "rowmax": online[1].clone(),
                    "rowsum": online[2].clone()}
            tables = (zt.clone(), ert.clone())
        else:
            table, gate = ex.gather_one(zd[r0:r1])
            outs = {"out": kernels.aggregate(part.local, table, part.permute_edges(ew[e0:e1]), exchange=gate).clone()}
            tables = (table.clone(),)
        steps.append((outs, tables, wants))
    torch.cuda.synchronize()
    res = {"bounds": np.asarray(part.bounds)}
    for s, (outs, tables, wants) in enumerate(steps):
        try:          # every slot of this rank's table held its owner's rows of that step after the launch
            assert_slots_hold([part], [(None, tables, None)], wants, f"{case} rank {rank} step {s + 1}")
            res[f"slots{s}"] = np.array("ok")
        except AssertionError as exc:
            res[f"slots{s}"] = np.array(str(exc))
        for k, v in outs.items():
            res[f"{k}{s}"] = v.float().cpu().numpy()
    return res


def _exec_case(case, rank, world, coo, host, gloo):
    """Four steps of one execute() case through a real exchange.  Returns {name: array}."""
    import torch
    from gta_graph_tensor_acclelrator_for_general_gnn_b200 import dist as gdist, executor
    isa, opg, network, reorder, exname, dt = EXEC_CASES[case]
    n = coo[0]
    fused = exname == "fused"

    def setup():
        p = _partition(host, n, rank, world, fused)
        return (p, gdist.FusedExchange(p) if fused else gdist.SourceExchange(p),
                _load(os.path.join("opgraph", opg + ".yaml")), _load(os.path.join("isa", isa + ".yaml")))
    part, ex, op_info, records = _agreed(setup, gloo, world)
    r0, r1 = part.row_begin, part.row_end
    e0, e1 = int(host.indptr[r0]), int(host.indptr[r1])
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    data = {}          # every data set on the device before the first step: no host copy between steps
    for d in set(STEPS):
        node_inputs, weights, edge_inputs = _exec_inputs(op_info, n, host.e, d)
        data[d] = ({k: t(v[r0:r1]) for k, v in node_inputs.items()}, {k: t(v) for k, v in weights.items()},
                   {k: part.permute_edges(t(v[e0:e1])) for k, v in edge_inputs.items()})
    torch.cuda.synchronize()
    outs = []
    for s, d in enumerate(STEPS):
        _skew(s, rank, world)
        out = executor.execute(records, op_info, part.local, *data[d],
                               network=network, is_reorder=reorder, check_shapes=False, source_table=ex,
                               feature_dtype=torch.bfloat16 if dt == "bf16" else torch.float32)
        (_, y), = out.items()
        outs.append(y.clone())
    torch.cuda.synchronize()
    res = {"bounds": np.asarray(part.bounds)}
    for s, y in enumerate(outs):
        res[f"out{s}"] = y.cpu().numpy()
    return res


def _worker(rank, world, port, out_dir):
    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    gloo = dist.new_group(backend="gloo")
    try:
        coos = {g: _graph_coo(g) for g in _graphs(world)}
        hosts = {g: _host_graph(*c) for g, c in coos.items()}
        for case in _kernel_cases(world) + [f"exec-{c}" for c in _exec_cases(world)]:
            gname = "crafted" if case.startswith("exec-") else case.split("-", 1)[0]
            try:
                if case.startswith("exec-"):
                    res = _exec_case(case[5:], rank, world, coos[gname], hosts[gname], gloo)
                else:
                    res = _kernel_case(case, rank, world, coos[gname], hosts[gname], gloo)
                np.savez(os.path.join(out_dir, f"{case}.r{rank}.npz"), **res)
            except Exception:
                with open(os.path.join(out_dir, f"{case}.r{rank}.err"), "w") as fh:
                    fh.write(traceback.format_exc())
                raise
            dist.barrier(group=gloo)
    finally:
        torch.cuda.synchronize()
        dist.destroy_process_group()


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


_RUNS = {}


@pytest.fixture(scope="module")
def runs(tmp_path_factory):
    """``run(world)``: the directory of that world's outputs; the ranks run once per world, the first time it is asked
    for.  Skipped when the box has fewer GPUs than ranks."""
    import torch
    import torch.multiprocessing as mp

    def run(world):
        if torch.cuda.device_count() < world:
            pytest.skip(f"{world} ranks need {world} GPUs, this box has {torch.cuda.device_count()}")
        if world not in _RUNS:
            _cabi.load()          # built once here, not by W children at the same time
            out = tmp_path_factory.mktemp(f"world{world}")
            try:          # join=True: no rank outlives the call; a failed rank is reported per case by _results
                mp.spawn(_worker, args=(world, _free_port(), str(out)), nprocs=world, join=True)
            except Exception:
                pass
            _RUNS[world] = (out,)
        return _RUNS[world][0]
    return run


def _results(out, case, world):
    errs = [open(out / f"{case}.r{r}.err").read() for r in range(world) if (out / f"{case}.r{r}.err").exists()]
    assert not errs, f"{case}: a rank failed:\n" + errs[0]
    missing = [r for r in range(world) if not (out / f"{case}.r{r}.npz").exists()]
    assert not missing, f"{case}: ranks {missing} wrote nothing (the spawn failed: see the captured output)"
    return [dict(np.load(out / f"{case}.r{r}.npz")) for r in range(world)]


def _check_bounds(res, host, world, n):
    bounds = [int(v) for v in res[0]["bounds"]]
    assert bounds == [int(v) for v in O.partition_bounds(host.indptr, world)]
    assert all(list(r["bounds"]) == bounds for r in res)
    assert bounds[0] == 0 and bounds[-1] == n and all(a <= b for a, b in zip(bounds, bounds[1:]))
    return bounds


def _cat(res, key, bounds):
    parts = [r[key] for r in res]
    assert [p.shape[0] for p in parts] == list(np.diff(bounds)), f"{key}: the ranks' rows do not tile [0, N)"
    return np.concatenate(parts)


_HOSTS = {}


def _host(gname):
    if gname not in _HOSTS:
        _HOSTS[gname] = _host_graph(*_graph_coo(gname))
    return _HOSTS[gname]


# ---- kernel-level cases ------------------------------------------------------------------------------------------------
KERNEL_RUNS = [(w, c) for w in WORLDS for c in _kernel_cases(w)]


@pytest.mark.parametrize("world,case", KERNEL_RUNS, ids=[f"world{w}-{c}" for w, c in KERNEL_RUNS])
def test_fused_exchange_kernels_on_real_ranks(runs, world, case):
    """Every rank's rows against fp64 at every step (bounded and want_stats path for GAT, with rowmax and rowsum), every
    slot of every rank's table after each step, step 4 against step 1, and every rank's output against the single-process
    emulation of the same partition, data and copy-CTA count, bit for bit."""
    import torch
    out = runs(world)
    gname, name = case.split("-", 1)[0], case.split("-copy")[0].split("-", 1)[1]
    call, copy_ctas = KERNEL_CALLS[name], int(case.rsplit("copy", 1)[1])
    H = _host(gname)
    res = _results(out, case, world)
    bounds = _check_bounds(res, H, world, H.n)
    if gname == "hub":
        assert any(b0 == b1 for b0, b1 in zip(bounds, bounds[1:])), f"bounds {bounds} leave every rank rows"
    owner = _owner_of_rows(bounds, H.n)
    keys = ("bounded", "online", "rowmax", "rowsum") if call[0] == "gat" else ("out",)
    for s in range(len(STEPS)):
        for r in res:
            assert str(r[f"slots{s}"]) == "ok", str(r[f"slots{s}"])
    for rank, r in enumerate(res):
        for k in keys:
            assert np.array_equal(r[f"{k}0"], r[f"{k}3"]), f"{case} rank {rank}: {k} of step 4 differs from step 1"
    # the emulation on this GPU checks the oracle too (_gat_step / _aggregate_step)
    parts, exs = emulated(H.full, world, copy_ctas)
    try:
        assert parts[0].bounds == bounds
        for s, d in enumerate(STEPS):
            what = f"world {world} {case} step {s + 1} (d{d})"
            if call[0] == "gat":
                emu = _gat_step(H, parts, exs, *_gat_data(call, d, owner), call[1], what)
                want = {"bounded": emu[0], "online": emu[1]}
            else:
                x = _inputs(("gcn", "multiprocess"), f"x{d}", (H.n, 64))
                ew = synthetic.gcn_edge_norm(H.indptr, H.indices)
                want = {"out": _aggregate_step(H, parts, exs, x, ew[:, None], None, ew, "f32", what)}
            for k, v in want.items():
                got = _cat(res, f"{k}{s}", bounds)
                assert np.array_equal(got, v.cpu().numpy()), f"{what}: {k} differs from the single-process emulation"
            if call[0] == "gat":          # the real ranks' rowmax / rowsum against fp64 (outputs: equal to the emulation's)
                z, el, er = _gat_data(call, d, owner)
                r64 = _gat_from_z(H.indptr, H.indices, z, el, er)
                np.testing.assert_allclose(_cat(res, f"rowmax{s}", bounds), r64["rowmax"], rtol=1e-6, atol=1e-6)
                np.testing.assert_allclose(_cat(res, f"rowsum{s}", bounds), r64["S"], rtol=2e-5)
    finally:
        release(exs)
    heads = call[3]
    if call[0] == "gat" and heads <= 32 and heads & (heads - 1) == 0:          # stale statistics must show
        data = {d: _gat_data(call, d, owner) for d in (0, 1, 2)}
        for prev, d in ((0, 1), (1, 2)):
            stale = _er_max_per_owner(data[prev][2], owner, world)
            assert _stale_bound_breaks(H.indptr, H.indices, owner, data[d][1], data[d][2], stale), \
                f"{case}: a bound from d{prev}'s statistics would not break d{d}"


# ---- execute() cases ---------------------------------------------------------------------------------------------------
EXEC_RUNS = [(w, c) for w in WORLDS for c in _exec_cases(w)]


def _emulate_execute(H, world, records, op_info, network, reorder, ins, dtype):
    """The kernel sequence execute() issues under a fused exchange, emulated on this GPU: every rank's execute() runs
    with its aggregation deferred (the GEMM has written slot 0 and published), then the deferred aggregations run in
    rank order into the outputs execute() returned.  GAT and GCN only: there the aggregation is the last op."""
    import torch
    from gta_graph_tensor_acclelrator_for_general_gnn_b200 import executor, kernels
    parts, exs = emulated(H.full, world)
    real = {"aggregate": kernels.aggregate, "gat_aggregate": kernels.gat_aggregate}
    pending = []

    def deferred(name, table_arg):
        def call(g, *a, **kw):
            t = a[table_arg]
            o = kernels.alloc_table(g.num_rows, int(t.shape[1]), t.device)
            pending.append((real[name], g, a, dict(kw, out=o)))
            return o
        return call
    node_inputs, weights, edge_inputs = ins
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    outs = []
    try:
        kernels.aggregate, kernels.gat_aggregate = deferred("aggregate", 0), deferred("gat_aggregate", 2)
        for p, ex in zip(parts, exs):
            r0, r1 = p.row_begin, p.row_end
            e0, e1 = int(H.indptr[r0]), int(H.indptr[r1])
            out = executor.execute(records, op_info, p.local, {k: t(v[r0:r1]) for k, v in node_inputs.items()},
                                   {k: t(v) for k, v in weights.items()},
                                   {k: p.permute_edges(t(v[e0:e1])) for k, v in edge_inputs.items()},
                                   network=network, is_reorder=reorder, check_shapes=False, source_table=ex,
                                   feature_dtype=torch.bfloat16 if dtype == "bf16" else torch.float32)
            (_, y), = out.items()
            outs.append(y)
    finally:
        kernels.aggregate, kernels.gat_aggregate = real["aggregate"], real["gat_aggregate"]
    assert len(pending) == world and all(y.data_ptr() == c[3]["out"].data_ptr() for y, c in zip(outs, pending))
    for fn, g, a, kw in pending:
        fn(g, *a, **kw)
    torch.cuda.synchronize()
    got = [y.cpu().numpy() for y in outs]
    release(exs)
    return got


@pytest.mark.parametrize("world,case", EXEC_RUNS, ids=[f"world{w}-{c}" for w, c in EXEC_RUNS])
def test_execute_on_real_ranks(runs, world, case):
    """A partitioned execute() of a golden program, 4 steps of different inputs: every rank's rows against the fp64 op
    graph, step 4 against step 1; under the fused exchange GAT and GCN against the emulation of the same kernel
    sequence bit for bit; under the NCCL all-gather (ascending source order, as on one GPU) GCN, DGN and PNA against
    single-GPU execute() bit for bit and GAT within tolerance (its bound comes from the gathered table, padding rows
    included, so its shift may differ in the last bits)."""
    import torch
    from gta_graph_tensor_acclelrator_for_general_gnn_b200 import executor
    out = runs(world)
    isa, opg, network, reorder, exname, dt = EXEC_CASES[case]
    H = _host("crafted")
    res = _results(out, f"exec-{case}", world)
    bounds = _check_bounds(res, H, world, H.n)
    for rank, r in enumerate(res):
        assert np.array_equal(r["out0"], r["out3"]), f"{case} rank {rank}: step 4 differs from step 1"
    op_info, records = _load(os.path.join("opgraph", opg + ".yaml")), _load(os.path.join("isa", isa + ".yaml"))
    sem = O.NETWORK_SEMANTICS.get((network, reorder), {})
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    for s, d in enumerate(STEPS[:3]):
        what = f"world {world} {case} step {s + 1} (d{d})"
        ins = _exec_inputs(op_info, H.n, H.e, d)
        got = _cat(res, f"out{s}", bounds)
        ref, scale = O.run_opgraph(op_info, H.indptr, H.indices, *ins, semantics=sem, stabilize=True,
                                   return_scale=True)
        (final,) = [p for p in range(len(op_info)) if not op_info[p]["OUTPUT"]["output_list"]]
        if dt == "bf16":
            _assert_bf16_close(got, ref[final], scale[final], what=what)
        else:
            assert_close_rowscale(got, ref[final], scale[final], what=what)
        if exname == "fused" and network in ("GAT", "GCN"):
            emu = np.concatenate(_emulate_execute(H, world, records, op_info, network, reorder, ins, dt))
            assert np.array_equal(got, emu), f"{what}: differs from the single-process emulation"
        if exname == "nccl":
            single = executor.execute(records, op_info, H.full, {k: t(v) for k, v in ins[0].items()},
                                      {k: t(v) for k, v in ins[1].items()}, {k: t(v) for k, v in ins[2].items()},
                                      network=network, is_reorder=reorder, check_shapes=False)[final].cpu().numpy()
            if network == "GAT":
                assert_close_rowscale(got, single.astype(np.float64), scale[final], what=what + " against one GPU")
            else:
                assert np.array_equal(got, single), f"{what}: differs from the single-GPU execute()"
