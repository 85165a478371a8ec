import os, sys, time, json
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'tests'))
from hivedscheduler_b200 import trace, _cabi
lib = _cabi.load_cuda_library()
out = {}
# C5: one ordered batch (health flips + gangs), single CTA (health events are global)
t = trace.trace_c5()
bc = trace.BatchContext(lib, t["config"], t["n_groups"], t["n_pods"], t["max_group_leaves"], t["max_group_pods"])
bc.set_all_nodes_healthy()
t0 = time.perf_counter(); bc.process(t["events"], 3 * 64 * len(t["events"]) + 4096); dt = time.perf_counter() - t0
out["C5"] = {"gangs": int(t["decision"].sum()), "events": len(t["events"]), "seconds_e2e": dt, "gangs_per_s": int(t["decision"].sum()) / dt,
             "hash": "%016x" % bc.result_hash()}
bc.close()
# C2: 10 000 one-GPU pods, 4 VCs
t = trace.trace_c2()
bc = trace.BatchContext(lib, t["config"], t["n_groups"], t["n_pods"], t["max_group_leaves"], t["max_group_pods"])
bc.set_all_nodes_healthy()
t0 = time.perf_counter(); bc.process(t["events"], 3 * 8 * len(t["events"]) + 4096); dt = time.perf_counter() - t0
out["C2"] = {"decisions": len(t["events"]), "seconds_e2e": dt, "decisions_per_s": len(t["events"]) / dt, "hash": "%016x" % bc.result_hash()}
bc.close()
# C4: call-by-call harness (includes the Python harness itself)
from importlib import util
spec = util.spec_from_file_location("g", os.path.join(ROOT, "tests", "golden", "make_trace_hashes.py")); g = util.module_from_spec(spec); spec.loader.exec_module(g)
t0 = time.perf_counter(); h, log, st = trace.run_c4_interactive(lib, **g.c4_kwargs(100000)); dt = time.perf_counter() - t0
out["C4"] = {"gangs": 100000, "calls": st["schedule_events"], "seconds_wall_incl_python_harness": dt, "gangs_per_s": 100000 / dt, "hash": "%016x" % h}
print(json.dumps(out, indent=1))
