#!/usr/bin/env python
"""API-level parity fuzz: random Schedule / AddAllocatedPod / DeleteAllocatedPod / DeleteUnallocatedPod calls and node
health flips on the reference's own test cluster (example/config/design, with its 46 pod specs), through the host
mirror of internal.SchedulerAlgorithm, on two implementations of include/hived.h in lock step.  After EVERY call the
results (bind info / victims / wait reason / error class), every cell's state, the order of every cluster view and the
hidden state that decides later calls (tests/hidden_state.py: free / bad-free / doomed-bad lists, the cell counters,
used-leaf maps, the groups of the cells, bad nodes and every group's placement) are compared.  A platform error
(the reference's panic) ends a run on both sides — the reference leaves its state undefined there.

    python tests/fuzz_api.py emu  [first_seed n_seeds n_ops]   device program (1-lane host emulation) vs oracle
    python tests/fuzz_api.py simt [first_seed n_seeds n_ops]   device program (32-lane SIMT emulation) vs oracle
    python tests/fuzz_api.py cuda [first_seed n_seeds n_ops]   libhived_cuda.so vs oracle (GPU box)

Environment: FUZZ_CLUSTER=synthetic (synthetic_fixture instead of the design config), FUZZ_MIX, FUZZ_RENAME and
FUZZ_FILTERING (the operation mix, see run_seed), FUZZ_JOBS=n (n worker processes; emulations only).
"""
import copy
import os
import random
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
import hidden_state  # noqa: E402
from conftest import snapshot_bytes  # noqa: E402
from golden_scenario import load_fixture  # noqa: E402
from hivedscheduler_b200 import _cabi  # noqa: E402
from hivedscheduler_b200 import algorithm as alg  # noqa: E402
from hivedscheduler_b200.config import new_config  # noqa: E402


def _call(fn):
    """('ok', value) | ('user', msg) | ('platform', None)"""
    try:
        return ("ok", fn())
    except alg.WebServerError as e:
        return ("user", getattr(e, "code", 400))
    except alg.PlatformError:
        return ("platform", None)


def _norm(psr):
    if psr.pod_bind_info is not None:
        return ("bind", psr.pod_bind_info)
    if psr.pod_preempt_info is not None:
        return ("preempt", sorted(p.uid for p in psr.pod_preempt_info["all_victims"]))
    return ("wait", psr.pod_wait_info["reason"])


def synthetic_fixture():
    """FUZZ_CLUSTER=synthetic: a small homogeneous 5-level forest in the shape of BASELINE's C3-C5 (GPU / HALF / NODE / RACK /
    POD: 3 x 3 x 4 nodes x 8 GPUs) with three VCs that hold POD-, RACK- and NODE-level cells and leave two racks to
    opportunistic pods, and 48 generated pod specs (1-2 members, 1-8 GPUs x 1-4 pods, priorities -1..5, typed and
    untyped, lazy preemption on half of them) — the same random API calls on a tree whose cells split and merge over
    three levels above the node."""
    from hivedscheduler_b200 import config as cfgmod
    levels = [("HALF", "B200", 4), ("NODE", "HALF", 2), ("RACK", "NODE", 4), ("POD", "RACK", 3)]
    vcs = {"vcA": [("POD", 1), ("POD.RACK", 1)], "vcB": [("POD.RACK", 2), ("POD.RACK.NODE", 2)], "vcC": [("POD.RACK", 1)]}
    cfg = cfgmod._synthetic(levels, 3, "NODE", vcs, "n%04d")
    rng = random.Random(20240911)
    pss = {}
    for i in range(48):
        members = [{"leafCellNumber": rng.choice([1, 2, 4, 8]), "podNumber": rng.choice([1, 1, 2, 3, 4])}]
        if rng.random() < 0.3:
            members.append({"leafCellNumber": rng.choice([1, 2, 4, 8]), "podNumber": rng.choice([1, 2])})
        pss["spec%02d" % i] = {
            "affinityGroup": {"members": members, "name": "sg%d" % i}, "gangReleaseEnable": False,
            "ignoreK8sSuggestedNodes": rng.random() < 0.3, "lazyPreemptionEnable": rng.random() < 0.5,
            "leafCellNumber": members[0]["leafCellNumber"], "leafCellType": "B200" if rng.random() < 0.7 else "",
            "pinnedCellId": "", "priority": rng.choice([-1, -1, 0, 1, 1, 2, 5]), "virtualCluster": rng.choice(["vcA", "vcB", "vcC"])}
    return {"design_config": cfg, "pss": pss}


def fixture():
    """The cluster FUZZ_CLUSTER names: "synthetic" (synthetic_fixture), else the reference's design config."""
    return synthetic_fixture() if os.environ.get("FUZZ_CLUSTER") == "synthetic" else load_fixture()


def run_seed(lib_a, lib_b, seed: int, n_ops: int, fx=None, verbose=False):
    """Returns None (no divergence) or a description of the first one."""
    fx = fx or fixture()
    rng = random.Random(seed)
    cfg = new_config(copy.deepcopy(fx["design_config"]))
    hs = [alg.HivedAlgorithm(cfg, lib=lib, max_groups=1024, max_pods=4096, max_group_leaves=128, max_group_pods=16)
          for lib in (lib_a, lib_b)]
    import ctypes as C
    for lib in (lib_a, lib_b):
        lib.hived_debug_view_hash.restype = C.c_uint64
        lib.hived_debug_view_hash.argtypes = [C.c_void_p]
    nodes = list(hs[0].node_names)
    healthy = {n: False for n in nodes}
    for n in nodes:
        for h in hs:
            h.setHealthyNode(n)
        healthy[n] = True
    spec_names = sorted(fx["pss"])
    allocated = []   # [(pod_a, pod_b)] bound pods (with bind-info annotations)
    preempting = []  # [(pod_a, pod_b)]
    serial = 0

    def both(op):
        ra, rb = _call(lambda: op(hs[0], 0)), _call(lambda: op(hs[1], 1))
        return ra, rb

    # the operation mix (defaults: the mix every committed seed number refers to).  FUZZ_MIX = "a,b,c": Schedule below a,
    # DeleteAllocatedPod below b, DeleteUnallocatedPod below c, node flaps above; FUZZ_RENAME = share of the gangs that
    # get one of six suffixed names (the rest re-use the spec's own name: more groups re-created under the same name)
    t_sched, t_del, t_unalloc = (float(x) for x in os.environ.get("FUZZ_MIX", "0.55,0.78,0.85").split(","))
    p_rename = float(os.environ.get("FUZZ_RENAME", "0.5"))
    try:
        for step in range(n_ops):
            r = rng.random()
            what = None
            if r < t_sched or not allocated:
                name = rng.choice(spec_names)
                spec = copy.deepcopy(fx["pss"][name])
                # gangs get a fresh name now and then, so that both new and further pods of a group occur
                if rng.random() < p_rename:
                    spec["affinityGroup"]["name"] = "%s-%d" % (spec["affinityGroup"]["name"], rng.randrange(6))
                serial += 1
                pods = [alg.Pod(name="p%d" % serial, namespace="fz", uid="u%d" % serial, annotations={}) for _ in range(2)]
                for p in pods:
                    p.annotations[alg.ANNOTATION_POD_SCHEDULING_SPEC] = alg.to_yaml(spec)
                # (Filtering-phase calls only with FUZZ_FILTERING=1: a Filtering-phase bind that lands on Reserved cells makes
                # the reference's incremental used-leaf counters drift from its leaf priorities, which the device program
                # derives its keys from — the one known divergence class, DESIGN.md section 2)
                filtering = os.environ.get("FUZZ_FILTERING") == "1" and rng.random() < 0.4
                phase = alg.FILTERING_PHASE if filtering else alg.PREEMPTING_PHASE
                sugg = nodes if rng.random() < 0.8 else [n for n in nodes if rng.random() < 0.7]
                what = "Schedule(%s [%s] as %s, %s)" % (name, spec["affinityGroup"]["name"], pods[0].uid, phase)
                ra, rb = both(lambda h, k: _norm(h.Schedule(pods[k], sugg, phase)))
                if ra != rb:
                    return "seed %d op %d %s: %r != %r" % (seed, step, what, ra, rb)
                if ra[0] == "platform":
                    return None
                if ra[0] == "ok" and ra[1][0] == "bind":
                    bound = [alg.new_binding_pod(pods[k], (ra, rb)[k][1][1]) for k in range(2)]
                    what = "AddAllocatedPod(%s = %s [%s] on %s %s)" % (pods[0].uid, name, spec["affinityGroup"]["name"], ra[1][1]["node"], ra[1][1]["leafCellIsolation"])
                    ra, rb = both(lambda h, k: h.AddAllocatedPod(bound[k]))
                    if ra != rb:
                        return "seed %d op %d %s: %r != %r" % (seed, step, what, ra, rb)
                    if ra[0] == "platform":
                        return None
                    allocated.append(tuple(bound))
                elif ra[0] == "ok" and ra[1][0] == "preempt" and phase == alg.PREEMPTING_PHASE:
                    preempting.append(tuple(pods))
            elif r < t_del:
                pair = allocated.pop(rng.randrange(len(allocated)))
                what = "DeleteAllocatedPod(%s)" % pair[0].uid
                ra, rb = both(lambda h, k: h.DeleteAllocatedPod(pair[k]))
                if ra != rb:
                    return "seed %d op %d %s: %r != %r" % (seed, step, what, ra, rb)
                if ra[0] == "platform":
                    return None
            elif r < t_unalloc and preempting:
                pair = preempting.pop(rng.randrange(len(preempting)))
                what = "DeleteUnallocatedPod(%s)" % pair[0].uid
                ra, rb = both(lambda h, k: h.DeleteUnallocatedPod(pair[k]))
                if ra != rb:
                    return "seed %d op %d %s: %r != %r" % (seed, step, what, ra, rb)
                if ra[0] == "platform":
                    return None
            else:
                n = rng.choice(nodes)
                healthy[n] = not healthy[n]
                what = "%s(%s)" % ("setHealthyNode" if healthy[n] else "setBadNode", n)
                ra, rb = both(lambda h, k: (h.setHealthyNode if healthy[n] else h.setBadNode)(n))
                if ra != rb:
                    return "seed %d op %d %s: %r != %r" % (seed, step, what, ra, rb)
                if ra[0] == "platform":
                    return None
            sa, sb = snapshot_bytes(hs[0]._lib, hs[0]._ctx), snapshot_bytes(hs[1]._lib, hs[1]._ctx)
            if sa != sb:
                return "seed %d op %d %s: cell states differ" % (seed, step, what)
            va, vb = (int(h._lib.hived_debug_view_hash(h._ctx)) for h in hs)
            if va != vb:
                return "seed %d op %d %s: the persisted order of a cluster view differs" % (seed, step, what)
            # (groups and pods by name: each mirror interns its own ids)
            d = hidden_state.diff(*(hidden_state.full(h._lib, h._ctx, h._groups.names, h._pods.names) for h in hs))
            if d:
                return "seed %d op %d %s: hidden state differs: %s" % (seed, step, what, d)
            if verbose:
                print(step, what, ra if what.startswith("Schedule") else "")
    finally:
        for h in hs:
            h.close()
    return None


def main():
    which = sys.argv[1] if len(sys.argv) > 1 else "emu"
    first = int(sys.argv[2]) if len(sys.argv) > 2 else 1
    count = int(sys.argv[3]) if len(sys.argv) > 3 else 20
    n_ops = int(sys.argv[4]) if len(sys.argv) > 4 else 300
    import subprocess
    import __graft_entry__ as g
    oracle = _cabi.load_library(g.build_oracle())
    if which == "cuda":
        lib = _cabi.load_cuda_library()
    else:
        src, out = {"emu": ("hived_emu.cpp", "libhived_emu.so"), "simt": ("hived_simt.cpp", "libhived_simt.so")}[which]
        path = os.path.join(HERE, "_build", out)
        os.makedirs(os.path.dirname(path), exist_ok=True)
        subprocess.check_call(["g++", "-O1", "-g", "-std=c++17", "-fPIC", "-shared", "-o", path, os.path.join(HERE, "emu", src)])
        lib = _cabi.load_library(path)
    global _JOB
    _JOB = (lib, oracle, n_ops, fixture())
    seeds = range(first, first + count)
    jobs = int(os.environ.get("FUZZ_JOBS", "1"))
    bad = 0
    if jobs > 1 and which != "cuda":
        import multiprocessing
        with multiprocessing.get_context("fork").Pool(jobs) as pool:  # workers inherit the loaded libraries
            results = list(pool.imap(_run_job, seeds, chunksize=4))
    else:
        results = map(_run_job, seeds)
    for d in results:
        if d:
            bad += 1
            print("DIVERGED", d, flush=True)
    cluster = "synthetic cluster" if os.environ.get("FUZZ_CLUSTER") == "synthetic" else "design config"
    print("api fuzz %s vs oracle on the %s: %d seeds x %d ops, %d divergences" % (which, cluster, count, n_ops, bad))
    return 1 if bad else 0


_JOB = None  # (lib_a, lib_b, n_ops, fixture) of main()


def _run_job(seed):
    lib_a, lib_b, n_ops, fx = _JOB
    return run_seed(lib_a, lib_b, seed, n_ops, fx)


if __name__ == "__main__":
    sys.exit(main())
