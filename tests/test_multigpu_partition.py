"""SURVEY.md section 8 row (e): one calm batch partitioned over several ranks (include/hived_multigpu.h), on the CPU
tier.  The DEVICE PROGRAM runs in the test-only emulation libraries (tests/emu); the protocol is the product's
(hivedscheduler_b200/dist.py + the engine's mg* entry points).  Witness: the chain hash over the merged results of
all ranks equals the hash of an ordinary single-context run and the oracle's, for every world size."""
import ctypes as C
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

from conftest import run_trace
from hivedscheduler_b200 import _cabi, dist, trace
from test_device_program_emu import small_c3

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _contexts(lib, t, world):
    out = []
    for _ in range(world):
        bc = trace.BatchContext(lib, t["config"], t["n_groups"], t["n_pods"], t["max_group_leaves"], t["max_group_pods"])
        bc.set_all_nodes_healthy()
        out.append(bc)
    return out


def simulate(lib, t, world, alloc=None, window=0):
    """`world` ranks in one process, the two collectives done by hand.  alloc(nbytes) -> (keepalive, pointer) of the
    exchange buffer (device memory for the CUDA library; default: host memory for the emulation libraries)."""
    dist.bind_multigpu(lib)
    ev = np.ascontiguousarray(t["events"])
    n = len(ev)
    evp = ev.ctypes.data_as(C.POINTER(_cabi.Event))
    cap = trace.pool_words_for(t)
    ranks = _contexts(lib, t, world)
    for r, bc in enumerate(ranks):
        assert lib.hived_mg_stage(bc.ctx, evp, n, cap, r, world) == 0, lib.hived_last_error(bc.ctx)
    nbytes = int(lib.hived_mg_shared_bytes(ranks[0].ctx))
    if alloc is None:
        buf = np.zeros(nbytes, dtype=np.uint8)
        buf_ptr = buf.ctypes.data
    else:
        buf, buf_ptr = alloc(nbytes)
    rounds = 0
    horizon = window if window > 0 else dist.DONE  # window = 0: the protocol without a horizon (hived_mg_run)
    while True:
        stops = []
        for bc in ranks:
            s = C.c_int32(0)
            if window > 0:
                assert lib.hived_mg_run_window(bc.ctx, min(horizon, dist.DONE), C.byref(s)) == 0, lib.hived_last_error(bc.ctx)
            else:
                assert lib.hived_mg_run(bc.ctx, C.byref(s)) == 0, lib.hived_last_error(bc.ctx)
            stops.append(s.value)
        e = min(stops)
        if e == dist.DONE:
            if horizon >= n:
                break
            horizon += window
            continue
        rounds += 1
        owner = stops.index(e)
        assert lib.hived_mg_solo(ranks[owner].ctx, e) == 0, lib.hived_last_error(ranks[owner].ctx)
        lib.hived_mg_export_shared(ranks[owner].ctx, C.c_void_p(buf_ptr))
        for r, bc in enumerate(ranks):
            if r != owner:
                lib.hived_mg_import_shared(bc.ctx, C.c_void_p(buf_ptr))
    fetched = []
    for bc in ranks:
        assert lib.hived_mg_finish(bc.ctx) == 0
        fetched.append(dist.fetch_results(lib, bc.ctx, n, cap))
    h = dist.chain_hash(lib, evp, n, world, [f[0].ctypes.data for f in fetched], [f[1].ctypes.data for f in fetched])
    # every SCHEDULE event was answered by exactly one rank
    sched = ev["type"] == _cabi.EV_SCHEDULE
    answered = sum(((f[0]["kind"] != 0) | (f[0]["wait_code"] != 0)).astype(np.int64) for f in fetched)
    assert answered[sched].max() <= 1
    for bc in ranks:
        bc.close()
    return h, rounds


@pytest.mark.parametrize("world,window", [(1, 0), (2, 0), (3, 0), (2, 64), (3, 7)])
def test_partitioned_simt_matches_single_run(simt_lib, oracle_lib, world, window):
    t = small_c3(400)
    h1, _, _ = run_trace(oracle_lib, t)
    h, rounds = simulate(simt_lib, t, world, window=window)
    assert h == h1
    assert rounds >= 1  # the first gang of each VC binds a preassigned cell


@pytest.fixture(scope="module")
def c3_8vc(oracle_lib):
    t = trace.trace_c3(n_gangs=1200)  # BASELINE configs[2]'s cluster (8192 nodes, 8 VCs), a short trace
    return t, run_trace(oracle_lib, t)[0]


@pytest.mark.parametrize("world,window", [(1, 0), (2, 0), (4, 0), (8, 0), (2, 256), (4, 100), (8, 1), (8, 1024)])
def test_partitioned_mt_matches_single_run_on_8_vcs(emu_mt_lib, c3_8vc, world, window):
    """window > 0: the horizon form of the protocol (hived_mg_run_window), what dist.run_partitioned drives."""
    t, h1 = c3_8vc
    h, rounds = simulate(emu_mt_lib, t, world, window=window)
    assert h == h1
    assert rounds >= 8


def test_partition_refuses_a_batch_that_is_not_calm(emu_mt_lib):
    lib = emu_mt_lib
    dist.bind_multigpu(lib)
    t = small_c3(50)
    bc = _contexts(lib, t, 1)[0]
    ev = np.ascontiguousarray(t["events"][:20]).copy()
    ev["type"][3] = _cabi.EV_NODE_HEALTH
    rc = lib.hived_mg_stage(bc.ctx, ev.ctypes.data_as(C.POINTER(_cabi.Event)), len(ev), 1 << 16, 0, 2)
    assert rc != 0 and b"SCHEDULE" in lib.hived_last_error(bc.ctx)
    bc.close()


WORKER = r'''
import ctypes as C, os, sys
sys.path.insert(0, %r); sys.path.insert(0, os.path.join(%r, "tests"))
import numpy as np
import torch.distributed as td
from hivedscheduler_b200 import _cabi, dist, trace
from test_device_program_emu import small_c3
rank, world, _ = dist.dist_env()
td.init_process_group("gloo", init_method="tcp://127.0.0.1:%%s" %% os.environ["MASTER_PORT"], rank=rank, world_size=world)
lib = _cabi.load_library(%r)
dist.bind_multigpu(lib)
t = small_c3(600)
bc = trace.BatchContext(lib, t["config"], t["n_groups"], t["n_pods"], t["max_group_leaves"], t["max_group_pods"])
bc.set_all_nodes_healthy()
ev = np.ascontiguousarray(t["events"]); n = len(ev); cap = trace.pool_words_for(t)
evp = ev.ctypes.data_as(C.POINTER(_cabi.Event))
info = dist.run_partitioned(lib, bc.ctx, evp, n, cap, rank, world, device="cpu")
res, pool, used = dist.fetch_results(lib, bc.ctx, n, cap)
gathered = [None] * world
td.all_gather_object(gathered, (res.tobytes(), pool[:used].tobytes()))
if rank == 0:
    rs = [np.frombuffer(g[0], dtype=trace.RESULT_DT) for g in gathered]
    ps = [np.frombuffer(g[1] + b"\0\0\0\0", dtype=np.int32) for g in gathered]
    h = dist.chain_hash(lib, evp, n, world, [r.ctypes.data for r in rs], [p.ctypes.data for p in ps])
    print("HASH %%016x rounds %%d" %% (h, info["rounds"]))
td.barrier()
td.destroy_process_group()
'''


def test_partitioned_over_gloo_world_size_2(emu_mt_lib, oracle_lib):
    t = small_c3(600)
    h1, _, _ = run_trace(oracle_lib, t)
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    src = WORKER % (ROOT, ROOT, emu_mt_lib._name)
    procs = []
    for rank in range(2):
        env = dict(os.environ, RANK=str(rank), WORLD_SIZE="2", LOCAL_RANK=str(rank), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        procs.append(subprocess.Popen([sys.executable, "-c", src], env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT))
    outs = [p.communicate(timeout=300)[0].decode() for p in procs]
    for p, o in zip(procs, outs):
        assert p.returncode == 0, o
    line = [l for l in outs[0].splitlines() if l.startswith("HASH")][0]
    assert int(line.split()[1], 16) == h1, line


def test_bench_partitioned_leg_plumbing_over_gloo(emu_mt_lib, oracle_lib):
    """bench.py --gpus 2 as the driver launches it (torch.distributed.run, one process per rank), on the emulation
    library under gloo: one JSON line from rank 0, strong scaling, the merged chain hash equal to the oracle's."""
    import json
    t = trace.trace_c3(n_gangs=1200)
    h1 = run_trace(oracle_lib, t)[0]
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    # bench.py takes the emulation path only without a visible GPU: hide any, so both ranks run it on every machine
    env = dict(os.environ, HIVED_BENCH_PLUMBING_TEST_LIB=emu_mt_lib._name, CUDA_VISIBLE_DEVICES="")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                          "--master-port", str(port), os.path.join(ROOT, "bench.py"), "--gpus", "2", "--steps", "1", "--warmup", "1",
                          "--gangs", "1200"], env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-3000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    line = json.loads(lines[0])
    assert line["n_gpus"] == 2 and line["scaling"] == "strong" and line["unit"] == "decisions/s"
    assert line["parity"]["result_hash"] == "%016x" % h1
    assert line["config"]["rounds_per_step"] >= 8 and line["e2e"]["value"] > 0
