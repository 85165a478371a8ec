#!/usr/bin/env python
"""bench.py — scheduling decisions/sec of the HiveD hot path on the BASELINE workload (C3).

A "step" is one pass of the hot path over the whole synthetic C3 trace (64k-GPU, 5-level cell tree,
8 VCs, 100 000 mixed gangs = 332 954 ordered events; SURVEY.md section 8d) starting from the same
cluster state.  ``value`` times the kernel with the batch already resident in HBM; ``e2e`` times the
reference-facing C-ABI call ``hived_process_events`` with pinned HOST buffers (H2D of the events and D2H
of the results inside the timed region).  ``--impl reference`` times the reference's own CPU algorithm
(the oracle: a faithful C++ restatement of the Go path; Go itself is not available in this image).

One JSON line is printed by rank 0.  ``--dump-outputs DIR`` also writes the results of the last timed step as .npy
files, so that two builds can be compared output for output on the same seeded trace.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the tree may be read-only: the benchmark writes nothing into it

from hivedscheduler_b200 import _cabi, trace  # noqa: E402

METRIC = "scheduling decisions/sec on 64k-GPU cell tree, 100k pending gangs"
# dram__bytes_read.sum + dram__bytes_write.sum of hived_events_kernel over the full C3 trace (one ncu --set full capture)
NCU_DRAM_BYTES_PER_LAUNCH_C3 = 88_998_912 + 93_801_728  # profiles/r2_final.md section 2 (the final kernel)
WORKLOAD = "C3: 8192 nodes x 8 GPU (65536 GPUs), 5-level tree, 8 VCs, 100000 mixed gangs (1/4/8/64-GPU), admission window 0.9"


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, device: int):
        super().__init__(daemon=True)
        self.device = device
        self.samples = []
        self.stop_flag = threading.Event()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag.is_set():
            try:
                out = subprocess.check_output(["nvidia-smi", "-i", str(self.device), "--query-gpu=" + q,
                                               "--format=csv,noheader,nounits"], timeout=5).decode().strip()
                self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = sorted(int(s[0]) for s in self.samples if s[0].isdigit())
        mx = max(int(s[1]) for s in self.samples if s[1].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(s[2 + i].lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": reasons, "samples": len(self.samples)}


def bind_bench_hooks(lib):
    P = C.c_void_p
    for name, res, args in [
        ("hived_bench_save_state", C.c_int, [P]), ("hived_bench_restore_state", C.c_int, [P]),
        ("hived_bench_stage_events", C.c_int, [P, C.POINTER(_cabi.Event), C.c_int32, C.c_int64]),
        ("hived_bench_run_staged", C.c_int, [P]),
        ("hived_bench_fetch_results", C.c_int, [P, C.POINTER(_cabi.Result), C.POINTER(C.c_int32), C.c_int64, C.POINTER(C.c_int64)]),
        ("hived_bench_flush_l2", C.c_int, [P]), ("hived_bench_phase_cycles", C.c_int, [P, C.POINTER(C.c_int64)]),
        ("hived_bench_last_kernel_ms", C.c_double, [P]),
        ("hived_bench_total_kernel_ms", C.c_double, [P]), ("hived_bench_kernel_launches", C.c_int64, [P]),
        ("hived_bench_num_ctas", C.c_int, [P]), ("hived_bench_set_result_hash", C.c_int, [P, C.c_int]),
        ("hived_bench_debug_cycles", C.c_int, [P, C.POINTER(C.c_int64)]),
        ("hived_bench_path_counters", C.c_int, [P, C.POINTER(C.c_int64)])]:
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args


DUMP_BUDGET_BYTES = 60_000_000  # array data of --dump-outputs; with the .npy headers the files stay under 64 MB


def dump_outputs(out_dir, res, pool):
    """What hived_process_events hands its caller for the batch: one float64 file per field of hived_result_t
    (result_<field>.npy, one row per event; int32 values are exact in float64) and the result pool (pool.npy).
    result_index.npy / pool_index.npy name the event rows and pool words written: all of them when they fit
    DUMP_BUDGET_BYTES, otherwise the same fixed seeded sample of both, sorted, for every run of the same trace."""
    os.makedirs(out_dir, exist_ok=True)
    cols = sum(int(np.prod(res.dtype[f].shape)) for f in res.dtype.names)
    rows, words = len(res), len(pool)
    values = rows * (cols + 1) + words * 2  # +1 / *2: the index arrays
    cap = DUMP_BUDGET_BYTES // 8
    rng = np.random.default_rng(0)

    def pick(n):
        k = n if values <= cap else int(n * cap / values)
        return np.arange(n) if k == n else np.sort(rng.choice(n, k, replace=False))

    ri, pi = pick(rows), pick(words)
    np.save(os.path.join(out_dir, "result_index.npy"), ri.astype(np.float64))
    for f in res.dtype.names:
        np.save(os.path.join(out_dir, "result_%s.npy" % f), res[f][ri].astype(np.float64))
    np.save(os.path.join(out_dir, "pool_index.npy"), pi.astype(np.float64))
    np.save(os.path.join(out_dir, "pool.npy"), pool[pi].astype(np.float64))


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def cpu_baseline(t, n_decisions: int, chunk_start: int = 0, ctx_holder=None):
    """The reference's CPU algorithm (oracle port) on a bounded sample of the same trace."""
    import __graft_entry__ as g
    lib = _cabi.load_library(g.build_oracle())
    if ctx_holder is None or "bc" not in ctx_holder:
        bc = trace.BatchContext(lib, t["config"], t["n_groups"], t["n_pods"], t["max_group_leaves"], t["max_group_pods"])
        bc.set_all_nodes_healthy()
        if ctx_holder is not None:
            ctx_holder["bc"] = bc
    else:
        bc = ctx_holder["bc"]
    dec = np.flatnonzero(t["decision"])
    lo = 0 if chunk_start == 0 else int(dec[chunk_start])
    hi = int(dec[chunk_start + n_decisions]) if chunk_start + n_decisions < len(dec) else len(t["events"])
    ev = t["events"][lo:hi]
    t0 = time.perf_counter()
    bc.process(ev, 3 * 64 * len(ev) + 4096)
    dt = time.perf_counter() - t0
    return n_decisions / dt, dt, len(ev)


def cpu_flat(t, max_threads: int = 8):
    """The DEVICE PROGRAM itself compiled for the host (-O2, tests/emu/hived_emu_mt.cpp): what the flat data structures
    and the algorithmic work of this repo give on CPU cores — 1 thread, and one thread per group of VCs with the same
    ordered shared sections as on the GPU.  Kernel-only time (events staged, results not fetched), like ``value``."""
    import __graft_entry__ as g
    lib = _cabi.load_library(g.build_cpu_flat())
    bind_bench_hooks(lib)
    ev = t["events"]
    n_dec = int(t["decision"].sum())
    pw = trace.pool_words_for(t)
    evp = ev.ctypes.data_as(C.POINTER(_cabi.Event))
    out = {"unit": "decisions/s", "what": "the device program compiled for the host (g++ -O2), 1-lane CTAs on host threads; "
                                          "kernel-only time over the whole C3 trace, best of 3"}
    nthreads = max(1, min(max_threads, os.cpu_count() or 1))
    for key, ncta in (("threads_1", 1), ("threads_n", nthreads)):
        os.environ["HIVED_NCTA"] = str(ncta)
        bc = trace.BatchContext(lib, t["config"], t["n_groups"], t["n_pods"], t["max_group_leaves"], t["max_group_pods"])
        bc.set_all_nodes_healthy()
        lib.hived_bench_save_state(bc.ctx)
        res, pool = bc.process(ev, pw)  # one pass through the ABI for the parity hash
        h = bc.result_hash()
        lib.hived_bench_stage_events(bc.ctx, evp, len(ev), pw)
        best = None
        for _ in range(3):
            lib.hived_bench_restore_state(bc.ctx)
            t0 = time.perf_counter()
            rc = lib.hived_bench_run_staged(bc.ctx)
            dt = time.perf_counter() - t0
            assert rc == 0, rc
            best = dt if best is None else min(best, dt)
        out[key] = {"value": n_dec / best, "threads": lib.hived_bench_num_ctas(bc.ctx), "seconds": best, "result_hash": "%016x" % h}
        bc.close()
    os.environ.pop("HIVED_NCTA", None)
    return out


def other_configs(lib):
    """BASELINE's other configurations on the GPU, end to end through the C ABI from host buffers, each checked against
    the oracle's committed hash (tests/golden/trace_hashes.json): C2 and C5 as one batch, C4 call by call (its event
    stream depends on the decisions: the harness plays kube-scheduler)."""
    golden = json.load(open(os.path.join(ROOT, "tests", "golden", "trace_hashes.json")))
    out = {}
    t = trace.trace_c2()
    bc = trace.BatchContext(lib, t["config"], t["n_groups"], t["n_pods"], t["max_group_leaves"], t["max_group_pods"])
    bc.set_all_nodes_healthy()
    # C2 is 10 000 events (about 40 ms): one cold pass is at the mercy of one-time costs of a fresh context (first
    # multi-CTA launch of it, page faults of the result buffers: 34 k - 250 k decisions/s from box to box), so the trace
    # runs three times from the same saved state and the line carries the best pass AND the first one
    lib.hived_bench_save_state(bc.ctx)
    times, h2 = [], None
    for i in range(3):
        if i:
            lib.hived_bench_restore_state(bc.ctx)
        t0 = time.perf_counter(); bc.process(t["events"], 3 * 8 * len(t["events"]) + 4096); times.append(time.perf_counter() - t0)
        if h2 is None:
            h2 = "%016x" % bc.result_hash()
    dt = min(times)
    out["C2"] = {"decisions_per_s": len(t["events"]) / dt, "seconds_e2e": dt, "seconds_e2e_first_pass": times[0],
                 "passes": "best of 3 from the same saved state", "result_hash": h2,
                 "matches_oracle": h2 == golden["C2"]["checkpoints"][-1]["hash"]}
    bc.close()
    t = trace.trace_c5()
    bc = trace.BatchContext(lib, t["config"], t["n_groups"], t["n_pods"], t["max_group_leaves"], t["max_group_pods"])
    bc.set_all_nodes_healthy()
    t0 = time.perf_counter(); bc.process(t["events"], 3 * 64 * len(t["events"]) + 4096); dt = time.perf_counter() - t0
    out["C5"] = {"gangs_per_s": int(t["decision"].sum()) / dt, "seconds_e2e": dt, "events": int(len(t["events"])),
                 "result_hash": "%016x" % bc.result_hash(),
                 "matches_oracle": "%016x" % bc.result_hash() == golden["C5"]["checkpoints"][-1]["hash"]}
    bc.close()
    from importlib import util
    spec = util.spec_from_file_location("mth", os.path.join(ROOT, "tests", "golden", "make_trace_hashes.py"))
    mth = util.module_from_spec(spec); spec.loader.exec_module(mth)
    # the closed loop played by compiled code (tests/harness/c4_player.cpp): every call goes through hived_process_events
    h, log, st, tm = trace.run_c4_compiled(lib, **mth.c4_kwargs(100000))
    c4_gpu = tm
    out["C4"] = {"gangs_per_s": 100000 / tm["seconds"], "seconds": tm["seconds"], "calls": tm["calls"], "events": tm["events"],
                 "us_per_call": 1e6 * tm["seconds"] / tm["calls"], "schedule_calls": int(st["schedule_events"]),
                 "harness": "compiled (c4_player.cpp), a gang's pod deletions as one batch",
                 "result_hash": "%016x" % h, "log_sha256_matches_oracle": mth.log_digest(log) == golden.get("C4", {}).get("log_sha256"),
                 "matches_oracle": "%016x" % h == golden.get("C4", {}).get("hash")}
    # the honest comparator for these configurations too: the DEVICE PROGRAM compiled for the host (cpu_flat, one thread:
    # C4 and C5 run on one CTA on the GPU as well; C2 on as many threads as CTAs), same calls, same hashes
    try:
        import __graft_entry__ as g
        flat = _cabi.load_library(g.build_cpu_flat())
        cf = {}
        for name, t_, pw in (("C2", trace.trace_c2(), lambda t: 3 * 8 * len(t["events"]) + 4096),
                             ("C5", trace.trace_c5(), lambda t: 3 * 64 * len(t["events"]) + 4096)):
            if name == "C5":
                os.environ["HIVED_NCTA"] = "1"
            bc = trace.BatchContext(flat, t_["config"], t_["n_groups"], t_["n_pods"], t_["max_group_leaves"], t_["max_group_pods"])
            bc.set_all_nodes_healthy()
            t0 = time.perf_counter(); bc.process(t_["events"], pw(t_)); dt = time.perf_counter() - t0
            os.environ.pop("HIVED_NCTA", None)
            units = len(t_["events"]) if name == "C2" else int(t_["decision"].sum())
            cf[name] = {"per_s": units / dt, "seconds": dt, "result_hash": "%016x" % bc.result_hash()}
            bc.close()
        h, log, st, tm = trace.run_c4_compiled(flat, **mth.c4_kwargs(100000))
        cf["C4"] = {"per_s": 100000 / tm["seconds"], "seconds": tm["seconds"], "us_per_call": 1e6 * tm["seconds"] / tm["calls"],
                    "result_hash": "%016x" % h}
        out["cpu_flat"] = dict(cf, what="the device program compiled for the host (g++ -O2), same calls; C2 on one thread per "
                                        "group of VCs, C4 / C5 on one thread (they run on one CTA on the GPU too)")
    except Exception as e:  # noqa  (a comparator must not take the bench line down)
        out["cpu_flat"] = {"unavailable": repr(e)}
    return out


def run_reference_arm(args):
    rank, world, _ = dist_env()
    if rank != 0:
        return
    t = trace.trace_c3()
    holder = {}
    sample = 400  # decisions per step: ~4 s of single-core work each
    for i in range(args.warmup):
        cpu_baseline(t, sample, i * sample, holder)
    t0 = time.perf_counter()
    done = 0
    for i in range(args.steps):
        cpu_baseline(t, sample, (args.warmup + i) * sample, holder)
        done += sample
    dt = time.perf_counter() - t0
    value = done / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "decisions/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / max(1, args.steps), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "int32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "sample": "%d consecutive decisions of the C3 trace per step" % sample},
        "cpu_baseline": {"value": value, "unit": "decisions/s", "cores": 1, "kind": "port",
                         "sample": "consecutive %d-decision windows of the C3 trace (whole-trace oracle run: 88 decisions/s, "
                                   "tests/golden/trace_hashes.json); the algorithm is serialised by one lock in the reference "
                                   "(hived_algorithm.go:185), so 1 core" % sample},
        "e2e": {"value": value, "unit": "decisions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def frontend_leg(lib, n_events: int = 24000, clients: int = 32):
    """The extender-shaped path (SURVEY.md section 8 row f4): the first `n_events` events of the C3 trace as filter
    calls / pod deletions through the pod state machine of include/hived_frontend.h.  Two shapes: (a) everything
    queued, then drained (one hived_process_events per max_batch events); (b) `clients` concurrent callers blocking in
    hived_fe_filter like HTTP handler threads, batches forming while the GPU is busy.  Parity: every pod must get the
    node and GPUs the plain batch path gives it."""
    import threading
    from hivedscheduler_b200 import frontend as fe_mod
    t = trace.trace_c3(n_gangs=max(2000, n_events // 2))
    ev = t["events"][:n_events]
    # the plain batch path: the reference answers
    bc0 = trace.BatchContext(lib, t["config"], t["n_groups"], t["n_pods"], t["max_group_leaves"], t["max_group_pods"])
    bc0.set_all_nodes_healthy()
    res0, pool0 = bc0.process(ev, trace.pool_words_for(t))
    bc0.close()
    want = {}
    pods, order, counters = {}, [], {}
    for i in range(len(ev)):
        e = ev[i]
        g = int(e["spec"]["group"])
        if e["type"] == _cabi.EV_SCHEDULE:
            j = counters.get(g, 0)
            counters[g] = j + 1
            uid = "g%d-%d" % (g, j)
            sp = e["spec"]
            ann = ("virtualCluster: vc%d\npriority: %d\nleafCellType: B200\nleafCellNumber: %d\naffinityGroup:\n  name: default/gang%d\n"
                   "  members:\n  - podNumber: %d\n    leafCellNumber: %d\n" % (sp["vc"], sp["priority"], sp["leaf_num"], g,
                                                                               sp["member_pod_num"][0], sp["member_leaf_num"][0]))
            pods[uid] = ann
            order.append(("filter", uid))
            r = res0[i]
            want[uid] = (int(r["node"]), tuple(int(pool0[r["this_off"] + 3 * k + 1]) for k in range(int(r["this_n"])))) if r["kind"] == 1 else None
        else:
            order.append(("delete", "g%d-%d" % (g, int(e["arg0"]))))

    def fresh(max_batch):
        bc = trace.BatchContext(lib, t["config"], t["n_groups"], t["n_pods"], t["max_group_leaves"], t["max_group_pods"])
        bc.set_all_nodes_healthy()
        f = fe_mod.FrontEnd(lib, bc.ctx, t["n_groups"], t["n_pods"], max_batch=max_batch)
        for uid, ann in pods.items():
            f.add_unbound_pod(uid, "default/" + uid, ann)
        return bc, f

    def check(answers):
        bad = 0
        for uid, r in answers.items():
            got = (int(r.node), tuple(r.leaf_index[:r.n_leaves])) if r.kind == fe_mod.FE_BIND else None
            bad += got != want[uid]
        return bad == 0

    out = {"events": len(ev), "filter_calls": len(pods)}
    # (a) queued, then drained
    bc, f = fresh(4096)
    t0 = time.perf_counter()
    tickets = {}
    for kind, uid in order:
        if kind == "filter":
            tickets[uid] = f.enqueue_filter(uid)
        else:
            f.delete_pod(uid)
    t1 = time.perf_counter()
    f.drain()
    t2 = time.perf_counter()
    answers = {uid: f.take(tk) for uid, tk in tickets.items()}
    st = f.stats()
    out["queued_then_drained"] = {"events_per_s": len(ev) / (t2 - t1), "drain_ms": 1e3 * (t2 - t1), "enqueue_ms": 1e3 * (t1 - t0),
                                  "drains": st["drains"], "largest_batch": st["largest_batch"], "matches_batch_path": check(answers)}
    f.close()
    bc.close()
    # (b) concurrent blocking callers; a pod's deletion is issued by the client that owns the pod's gang (order within
    # a gang preserved; across gangs the arrival order is whatever the threads produce: parity is not defined, only
    # that no GPU is handed out twice)
    bc, f = fresh(4096)
    per = [[] for _ in range(clients)]
    for kind, uid in order:
        per[int(uid[1:].split("-")[0]) % clients].append((kind, uid))
    answers = {}

    def client(items):
        for kind, uid in items:
            if kind == "filter":
                answers[uid] = f.filter(uid)
            else:
                f.delete_pod(uid)

    ths = [threading.Thread(target=client, args=(items,)) for items in per]
    t0 = time.perf_counter()
    for th in ths:
        th.start()
    for th in ths:
        th.join()
    f.drain()
    dt = time.perf_counter() - t0
    st = f.stats()
    binds = sum(1 for r in answers.values() if r.kind == fe_mod.FE_BIND)
    out["concurrent_clients"] = {"clients": clients, "events_per_s": len(ev) / dt, "us_per_filter_call": 1e6 * dt / max(1, len(pods)),
                                 "drains": st["drains"], "mean_batch": st["events"] / max(1, st["drains"]), "largest_batch": st["largest_batch"],
                                 "bind_answers": binds, "note": "Python client threads (GIL): a lower bound for a Go / C++ extender"}
    f.close()
    bc.close()
    return out


def main_partitioned(args, lib, rank, world, local):
    """N > 1: ONE C3 batch partitioned over the ranks by virtual cluster (include/hived_multigpu.h; strong scaling:
    the total work is fixed).  Every rank holds the whole cluster; the result of the job is the merged results."""
    import torch
    import torch.distributed as dist
    from hivedscheduler_b200 import dist as hd
    hd.bind_multigpu(lib)
    on_gpu = torch.cuda.is_available()  # (False only in the gloo plumbing test of tests/test_multigpu_partition.py)
    t = trace.trace_c3(n_gangs=args.gangs)
    ev = t["events"]
    n = len(ev)
    n_dec = int(t["decision"].sum())
    pool_words = trace.pool_words_for(t)
    bc = trace.BatchContext(lib, t["config"], t["n_groups"], t["n_pods"], t["max_group_leaves"], t["max_group_pods"], device=local)
    bc.set_all_nodes_healthy()
    ctx = bc.ctx
    lib.hived_bench_save_state(ctx)
    ev_pinned = torch.empty(ev.nbytes, dtype=torch.uint8, pin_memory=on_gpu)
    ev_pinned.numpy()[:] = ev.view(np.uint8)
    ev_ptr = C.cast(ev_pinned.data_ptr(), C.POINTER(_cabi.Event))
    res_pinned = torch.empty(n * C.sizeof(_cabi.Result), dtype=torch.uint8, pin_memory=on_gpu)
    pool_pinned = torch.empty(pool_words, dtype=torch.int32, pin_memory=on_gpu)
    res_ptr = C.cast(res_pinned.data_ptr(), C.POINTER(_cabi.Result))
    pool_ptr = C.cast(pool_pinned.data_ptr(), C.POINTER(C.c_int32))
    device = "cuda:%d" % local if on_gpu else "cpu"
    used = C.c_int64()

    def barrier():
        dist.barrier()
        if on_gpu:
            torch.cuda.synchronize()

    info = {}

    def step(e2e: bool):
        lib.hived_bench_restore_state(ctx)
        lib.hived_bench_flush_l2(ctx)
        if not e2e:
            assert lib.hived_mg_reset(ctx) == 0
        barrier()
        k0 = lib.hived_bench_total_kernel_ms(ctx)
        if on_gpu:
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
        t0 = time.perf_counter()
        info.update(hd.run_partitioned(lib, ctx, ev_ptr, n, pool_words, rank, world, device=device, staged=not e2e))
        if e2e:
            assert lib.hived_bench_fetch_results(ctx, res_ptr, pool_ptr, pool_words, C.byref(used)) == 0
        if on_gpu:
            b.record()
            torch.cuda.synchronize()
        info["kernel_ms"] = lib.hived_bench_total_kernel_ms(ctx) - k0
        return a.elapsed_time(b) / 1e3 if on_gpu else time.perf_counter() - t0

    assert lib.hived_mg_stage(ctx, ev_ptr, n, pool_words, rank, world) == 0, lib.hived_last_error(ctx)
    for _ in range(args.warmup):
        step(False)
    sampler = ClockSampler(local)
    if on_gpu:
        sampler.start()
    launches0 = lib.hived_bench_kernel_launches(ctx)
    res_s = [step(False) for _ in range(args.steps)]
    launches = lib.hived_bench_kernel_launches(ctx) - launches0
    kernel_ms, coll_s, rounds = info["kernel_ms"], info["collective_s"], info["rounds"]
    for _ in range(min(args.warmup, 2)):
        step(True)
    e2e_s = [step(True) for _ in range(args.steps)]
    sampler.stop_flag.set()
    if on_gpu:
        sampler.join(timeout=2)
    times = torch.tensor([sum(res_s), sum(e2e_s), kernel_ms / 1e3, coll_s], dtype=torch.float64, device=device)
    dist.all_reduce(times, op=dist.ReduceOp.MAX)
    tot_s, tot_e2e, kernel_s_last, coll_s_last = [float(x) for x in times.tolist()]
    # parity witness: the chain hash over the merged results of the last (e2e) step
    res = np.frombuffer(res_pinned.numpy(), dtype=trace.RESULT_DT)
    gathered = [None] * world
    dist.all_gather_object(gathered, (res.tobytes(), pool_pinned.numpy()[:max(int(used.value), 1)].tobytes()))
    if rank == 0:
        rs = [np.frombuffer(g[0], dtype=trace.RESULT_DT) for g in gathered]
        ps = [np.frombuffer(g[1], dtype=np.int32) for g in gathered]
        h = hd.chain_hash(lib, ev_ptr, n, world, [r.ctypes.data for r in rs], [p_.ctypes.data for p_ in ps])
        peak, peak_src = measured_peak_gbs()
        stats = bc.stats()
        line = {
            "metric": METRIC, "value": n_dec * args.steps / tot_s, "unit": "decisions/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * tot_s / args.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "int32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "events_per_step": int(n), "decisions_per_step": n_dec,
                       "parallelism": "VC partition: rank r owns the VCs v %% %d == r, one CTA per owned VC; events that touch the "
                                      "chain-wide free lists run alone, in batch order (include/hived_multigpu.h)" % world,
                       "l2": "flushed between steps (256 MiB memset)",
                       "timing": "CUDA events on the torch stream around the whole partitioned pass (kernels + NCCL rounds); max over ranks",
                       "rounds_per_step": rounds, "broadcast_bytes_per_round": info["shared_bytes"],
                       "horizon_window_events": info.get("window"), "horizon_advances_per_step": info.get("windows"),
                       "slowest_rank_kernel_ms_last_step": 1e3 * kernel_s_last, "slowest_rank_collective_ms_last_step": 1e3 * coll_s_last,
                       "e2e": "hived_mg_stage from pinned host memory (H2D of the whole batch on every rank), the partitioned pass, "
                              "D2H of the rank's results + pool"},
            "e2e": {"value": n_dec * args.steps / tot_e2e, "unit": "decisions/s", "h2d_bytes_per_step": int(ev.nbytes) * world,
                    "d2h_bytes_per_step": int(n * C.sizeof(_cabi.Result)) * world},
            "gpu_launches": int(launches) * world,
            "clocks": sampler.summary() if on_gpu else None,
            "roofline": {"bound": "hbm", "achieved": stats["algorithmic_bytes"] / (tot_s / args.steps) / 1e9 * world, "peak": peak * world,
                         "unit": "GB/s", "frac": stats["algorithmic_bytes"] / (tot_s / args.steps) / 1e9 / peak, "traffic": None,
                         "kernel": "hived_events_kernel", "peak_source": peak_src,
                         "note": "rank 0's algorithmic bytes x ranks; the pass is latency-bound (DESIGN.md section 4)"},
            "parity": {"result_hash": "%016x" % h, "note": "chain hash over the merged results of all ranks"},
        }
        print(json.dumps(line))
    dist.barrier()
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--gangs", type=int, default=100000, help="C3 trace length (BASELINE: 100000)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--replicas", action="store_true", help="N > 1: independent replicas (weak scaling) instead of the VC partition")
    ap.add_argument("--no-other-configs", action="store_true", help="skip the C2 / C4 / C5 sub-lines (about 45 s)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the results of the last timed step to DIR/<name>.npy (float64, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and (args.impl == "reference" or (dist_env()[1] > 1 and not args.replicas)):
        ap.error("--dump-outputs writes the results of one whole batch: --impl ours on one GPU or with --replicas")
    if args.impl == "reference":
        return run_reference_arm(args)

    import torch
    import torch.distributed as dist
    rank, world, local = dist_env()
    emu = os.environ.get("HIVED_BENCH_PLUMBING_TEST_LIB")  # tests only: the N > 1 plumbing under gloo, on the emulation library
    if emu and world > 1 and not torch.cuda.is_available():
        dist.init_process_group("gloo")
        lib = _cabi.load_library(emu)
        bind_bench_hooks(lib)
        return main_partitioned(args, lib, rank, world, local)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    lib = _cabi.load_cuda_library()
    bind_bench_hooks(lib)
    if world > 1 and not args.replicas:
        return main_partitioned(args, lib, rank, world, local)

    t = trace.trace_c3(n_gangs=args.gangs)
    ev = t["events"]
    n_dec = int(t["decision"].sum())
    pool_words = trace.pool_words_for(t)
    bc = trace.BatchContext(lib, t["config"], t["n_groups"], t["n_pods"], t["max_group_leaves"], t["max_group_pods"], device=local)
    bc.set_all_nodes_healthy()
    ctx = bc.ctx
    lib.hived_bench_save_state(ctx)

    # pinned host buffers for the e2e leg
    ev_pinned = torch.empty(ev.nbytes, dtype=torch.uint8, pin_memory=True)
    ev_pinned.numpy()[:] = ev.view(np.uint8)
    res_pinned = torch.empty(len(ev) * C.sizeof(_cabi.Result), dtype=torch.uint8, pin_memory=True)
    pool_pinned = torch.empty(pool_words, dtype=torch.int32, pin_memory=True)
    ev_ptr = C.cast(ev_pinned.data_ptr(), C.POINTER(_cabi.Event))
    res_ptr = C.cast(res_pinned.data_ptr(), C.POINTER(_cabi.Result))
    pool_ptr = C.cast(pool_pinned.data_ptr(), C.POINTER(C.c_int32))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step_resident():
        lib.hived_bench_restore_state(ctx)
        lib.hived_bench_flush_l2(ctx)
        rc = lib.hived_bench_run_staged(ctx)
        assert rc == 0, rc
        return lib.hived_bench_last_kernel_ms(ctx)

    def step_e2e():
        lib.hived_bench_restore_state(ctx)
        lib.hived_bench_flush_l2(ctx)
        t0 = time.perf_counter()
        rc = lib.hived_process_events(ctx, ev_ptr, len(ev), None, 0, res_ptr, pool_ptr, pool_words)
        assert rc == 0, rc
        return time.perf_counter() - t0

    # ---- resident leg (value)
    lib.hived_bench_stage_events(ctx, ev_ptr, len(ev), pool_words)
    for _ in range(args.warmup):
        step_resident()
    sampler = ClockSampler(local)
    sampler.start()
    launches0 = lib.hived_bench_kernel_launches(ctx)
    barrier()
    t0 = time.perf_counter()
    kernel_ms = [step_resident() for _ in range(args.steps)]
    barrier()
    wall = time.perf_counter() - t0
    launches = lib.hived_bench_kernel_launches(ctx) - launches0
    n_ctas = lib.hived_bench_num_ctas(ctx)
    # parity witness: the hash of the last step's results
    used = C.c_int64()
    rc = lib.hived_bench_fetch_results(ctx, res_ptr, pool_ptr, pool_words, C.byref(used))
    assert rc == 0, rc
    if args.dump_outputs:  # copies: the legs below reuse the pinned buffers
        last_res = np.frombuffer(res_pinned.numpy(), dtype=trace.RESULT_DT).copy()
        last_pool = pool_pinned.numpy()[:used.value].copy()
    stats = bc.stats()
    cyc = (C.c_int64 * 15)()
    lib.hived_bench_phase_cycles(ctx, cyc)
    dbg = (C.c_int64 * 16)()
    lib.hived_bench_debug_cycles(ctx, dbg)
    pathc = (C.c_int64 * 16)()
    n_pathc = lib.hived_bench_path_counters(ctx, pathc)
    # the restore + L2 flush between steps are not part of a step: time = sum of the kernels' CUDA-event times
    kernel_total_s = sum(kernel_ms) / 1e3
    # ---- e2e leg
    # (the library's running FNV parity hash is test instrumentation, ~4 CPU cycles per result byte: off while timing)
    lib.hived_bench_set_result_hash(ctx, 0)
    for _ in range(min(args.warmup, 2)):
        step_e2e()
    e2e_times = [step_e2e() for _ in range(args.steps)]
    sampler.stop_flag.set()
    sampler.join(timeout=2)
    e2e_s = sum(e2e_times)
    # parity witness: one more (untimed) pass through the same call with the hash on
    lib.hived_bench_set_result_hash(ctx, 1)
    step_e2e()
    parity_hash = bc.result_hash()
    # ---- per-call leg: the extender's own pattern, one pod per call (one request / result round trip each):
    # the first events of the same trace through hived_process_events(n=1) — the same path hived_schedule takes
    lib.hived_bench_restore_state(ctx)
    lib.hived_bench_set_result_hash(ctx, 0)
    n_calls = min(3000, len(ev))
    one = C.sizeof(_cabi.Event)
    base = ev_pinned.data_ptr()
    for i in range(64):  # warm-up calls (also part of the sequence)
        lib.hived_process_events(ctx, C.cast(base + i * one, C.POINTER(_cabi.Event)), 1, None, 0, res_ptr, pool_ptr, pool_words)
    k0 = lib.hived_bench_total_kernel_ms(ctx)
    t0 = time.perf_counter()
    for i in range(64, n_calls):
        rc = lib.hived_process_events(ctx, C.cast(base + i * one, C.POINTER(_cabi.Event)), 1, None, 0, res_ptr, pool_ptr, pool_words)
        assert rc == 0, rc
    per_call_s = (time.perf_counter() - t0) / max(1, n_calls - 64)
    per_call_kernel_us = 1e3 * (lib.hived_bench_total_kernel_ms(ctx) - k0) / max(1, n_calls - 64)
    lib.hived_bench_set_result_hash(ctx, 1)

    times = torch.tensor([kernel_total_s, e2e_s, wall], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    kernel_total_s, e2e_s, wall = [float(x) for x in times.tolist()]
    value = world * n_dec * args.steps / kernel_total_s
    e2e_value = world * n_dec * args.steps / e2e_s
    peak, peak_src = measured_peak_gbs()
    # the device-side work counters are rewound with the state, so they describe ONE pass of the trace
    alg_bytes = stats["algorithmic_bytes"]
    achieved = alg_bytes / (kernel_total_s / args.steps) / 1e9
    line = {
        "metric": METRIC, "value": value, "unit": "decisions/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * kernel_total_s / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "int32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "events_per_step": int(len(ev)), "decisions_per_step": n_dec,
                   "parallelism": ("replicas" if world > 1 else "1 GPU") + ", %d CTAs (one per group of VCs)" % n_ctas, "l2": "flushed between steps (256 MiB memset)",
                   "timing": "CUDA events on the launch stream around the kernel; max over ranks",
                   "e2e": "hived_process_events from pinned host buffers (H2D events, kernel, pool compaction, D2H results + pool); "
                          "the library's running parity hash is switched off while timing and checked on an extra pass",
                   "wall_ms_per_step_incl_state_rewind": 1e3 * wall / args.steps},
        "e2e": {"value": e2e_value, "unit": "decisions/s", "h2d_bytes_per_step": int(ev.nbytes),
                "d2h_bytes_per_step": int(len(ev) * C.sizeof(_cabi.Result) + 4 * used.value)},
        "per_call": {"us_per_event": 1e6 * per_call_s, "kernel_us_per_event": per_call_kernel_us, "events": int(n_calls - 64),
                     "resident_kernel": os.environ.get("HIVED_NO_RESIDENT", "0") in ("", "0"),
                     "note": "hived_process_events with n=1 on the first events of the same trace, from Python: the latency the "
                             "HTTP extender sees per Schedule/Delete.  Served by the resident per-call kernel (request slot in "
                             "mapped host memory, no launch / memcpy / stream sync per call); HIVED_NO_RESIDENT=1 = one launch "
                             "per call.  From C: profiles/micro/percall_latency.c"},
        "gpu_launches": int(launches),
        "clocks": sampler.summary(),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": NCU_DRAM_BYTES_PER_LAUNCH_C3 if args.gangs == 100000 else None,
                     "traffic_source": "ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum of one full-size launch "
                                       "(profiles/r2_final.md section 2); bytes per launch",
                     "algorithmic_bytes_per_launch": int(alg_bytes), "kernel": "hived_events_kernel",
                     "peak_source": peak_src,
                     "note": "latency-bound sequential contract: the state (~9 MB of cells) is L2/L1 resident, DRAM traffic is "
                             "the event stream in and the results out; see DESIGN.md section 4"},
    }
    if rank == 0:
        if not args.no_cpu_baseline and world == 1:
            v, dt, nev = cpu_baseline(t, 1500)
            line["cpu_baseline"] = {"value": v, "unit": "decisions/s", "cores": 1, "kind": "port",
                                    "sample": "first 1500 decisions (%d events) of the same C3 trace, %.1f s" % (nev, dt)}
        if not args.no_cpu_baseline and world == 1:
            line["cpu_flat"] = cpu_flat(t)
        if not args.no_other_configs and world == 1 and args.gangs == 100000:
            line["other_configs"] = other_configs(lib)
            line["frontend"] = frontend_leg(lib)
        line["parity"] = {"result_hash": "%016x" % parity_hash}
        pc_names = ["view_bucketed", "view_full_pass", "bucket_rebuilds", "bucket_moves", "commit_lean", "commit_general",
                    "release_lean", "release_general", "map_lean", "map_general", "pod_of_gang_lean", "delete_pod_lean"]
        line["paths_per_step"] = {n: int(pathc[i]) for i, n in enumerate(pc_names[:n_pathc])}
        names = ["view_pass", "leaf_search", "map_v2p", "emit_result", "commit", "delete", "all_events", "shared_wait", "shared_sections",
                 "schedule_pod_of_existing_gang", "n_schedule_pod_of_existing_gang", "delete_not_last_pod", "n_delete_not_last_pod",
                 "commit_pod_of_existing_gang", "n_commit_pod_of_existing_gang"]
        if any(int(c) for c in cyc):  # SM-cycle counters exist in profiling builds only (HIVED_PROFILE=1 at build time)
            line["phase_cycles_per_step"] = {n: int(c) for n, c in zip(names, cyc)}
        if os.environ.get("HIVED_BENCH_DEBUG"):
            line["debug_cycles"] = [int(x) for x in dbg]
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, last_res, last_pool)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
