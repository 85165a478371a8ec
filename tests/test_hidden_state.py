"""The state that decides LATER calls — free / bad-free / doomed-bad lists in slice order, the cell counters, the
used-leaf maps with their drift, the groups of the cells (ghost records included), the bad nodes and every group's
placement (tests/hidden_state.py) — compared with the oracle at the end of every chunk of the trace families, after
the C4 harness's calls, and after every call of the API fuzz (tests/fuzz_api.py compares it for every seed, so the
regression seeds of test_device_program_emu.py / test_gpu_parity.py check it too).  A difference in this state shows
up in a result or a cell snapshot only many operations later, if at all."""
import os
import pickle
import subprocess
import sys

import pytest

import hidden_state
from conftest import run_trace
from hivedscheduler_b200 import config, trace
from test_device_program_emu import small_c3, small_cluster

HERE = os.path.dirname(os.path.abspath(__file__))

TRACES = {
    "C1": trace.trace_c1, "C2": lambda: trace.trace_c2(n_pods=700), "C3-small": lambda: small_c3(500),
    "multi-member": lambda: trace.trace_multi_member(n_gangs=300),
    "heterogeneous": lambda: trace.trace_heterogeneous(n_gangs=500),
    "suggested-nodes": lambda: trace.trace_suggested_nodes(n_gangs=250), "bad-requests": trace.trace_bad_requests,
    "C5-churn": lambda: trace.trace_c5(n_steps=4, gangs_per_step=300, n_nodes=4 * 16 * 32, n_vcs=2,
                                       vc_gpus=(16 + 6) * 32 * 8, config=small_cluster()),
}
C4 = dict(config=None, n_gangs=1200, n_vcs=2, vc_gpus=(16 + 6) * 32 * 8, total_gpus=4 * 16 * 32 * 8)
C4_LAZY = dict(C4, n_gangs=4500, lazy_percent=50, load=3.0)


def record_states(monkeypatch, every=1, ctas=None):
    """Patches trace.BatchContext to append the hidden state (hidden_state.full) after every `every`-th batch and
    before the context is closed; returns the list it appends to.  `ctas` (a list) receives the number of CTAs every
    batch ran on."""
    states, calls = [], [0]
    process, close = trace.BatchContext.process, trace.BatchContext.close

    def recording_process(self, *a, **kw):
        out = process(self, *a, **kw)
        calls[0] += 1
        if ctas is not None:
            ctas.append(self.lib.hived_bench_num_ctas(self.ctx))
        if calls[0] % every == 0:
            states.append(hidden_state.full(self.lib, self.ctx))
        return out

    def recording_close(self):
        if self.ctx:
            states.append(hidden_state.full(self.lib, self.ctx))
        close(self)

    monkeypatch.setattr(trace.BatchContext, "process", recording_process)
    monkeypatch.setattr(trace.BatchContext, "close", recording_close)
    return states


def assert_same_states(a, b):
    assert len(a) == len(b) and a, (len(a), len(b))
    for i, (x, y) in enumerate(zip(a, b)):
        d = hidden_state.diff(x, y, ("device", "oracle"))
        assert d is None, "after batch %d of %d: %s" % (i + 1, len(a), d)


def trace_states(lib, t, monkeypatch, chunks=3):
    states = record_states(monkeypatch)
    h, _, st = run_trace(lib, t, chunks=chunks)
    monkeypatch.undo()
    return h, st, states


def check_trace(lib, oracle, name, monkeypatch):
    t = TRACES[name]()
    ha, sa, a = trace_states(lib, t, monkeypatch)
    hb, sb, b = trace_states(oracle, t, monkeypatch)
    assert ha == hb and sa == sb
    assert_same_states(a, b)
    return a


def check_c4(lib, oracle, kw, monkeypatch):
    kw = dict(kw, config=small_cluster())
    out = []
    for x in (lib, oracle):
        states = record_states(monkeypatch, every=250)
        out.append(trace.run_c4_interactive(x, **kw) + (states,))
        monkeypatch.undo()
    (ha, la, sa, a), (hb, lb, sb, b) = out
    assert la == lb and ha == hb and sa == sb
    assert_same_states(a, b)
    return sb


def run_fuzz_seed(lib, oracle, seed, monkeypatch, **env):
    import fuzz_api
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    return fuzz_api.run_seed(lib, oracle, seed, 300)


SYNTHETIC_NO_RENAME_FILTERING = dict(FUZZ_CLUSTER="synthetic", FUZZ_RENAME="0.0", FUZZ_FILTERING="1")


# ---------------------------------------------------------------------------------------------------- the helpers


def test_decode_and_diff_name_the_first_differing_item():
    H = hidden_state
    words = [H.FREE, 0, 3, 3, 517, 518, 519, H.FREE, 1, 1, 1, 4, H.DOOMED_BAD, 2, 0, 4, 1, 399,
             H.VC_FREE, 0, 0, 5, -1, H.TOTAL_LEFT, 0, 5, 2, H.USED_PHYSICAL, 7, 2, -2, -1, 0, 8,
             H.USED_VIRTUAL, 3, 1, 1, 4, H.USING_GROUP, 9, 12, 1, H.RESERVING_GROUP, 9, 40, 0, H.BAD_NODE, 6]
    a = H.decode(words)
    assert a[(H.FREE, 0, 3)] == (517, 518, 519)
    assert a[(H.DOOMED_BAD, 2, 0, 4)] == (399,)
    assert a[(H.VC_FREE, 0, 0, 5)] == -1
    assert a[(H.USED_PHYSICAL, 7)] == ((-2, -1), (0, 8))
    assert a[(H.RESERVING_GROUP, 9)] == (40, 0)
    assert a[(H.BAD_NODE, 6)] is True
    assert H.diff(a, dict(a)) is None
    swapped = list(words)
    swapped[5], swapped[6] = swapped[6], swapped[5]
    assert H.diff(a, H.decode(swapped)) == "freeCellList[chain 0][level 3] position 1: 518 != 519"
    shorter = dict(a)
    shorter[(H.DOOMED_BAD, 2, 0, 4)] = (399, 401)
    assert H.diff(a, shorter).startswith("vcDoomedBadCells[vc 2][chain 0][level 4] length: 1 != 2")
    drift = dict(a)
    drift[(H.USED_PHYSICAL, 7)] = ((0, 8),)
    assert H.diff(a, drift) == "physical usedLeafCellNumAtPriorities of cell 7: {-2: -1, 0: 8} != {0: 8}"
    ghost = dict(a)
    ghost[(H.RESERVING_GROUP, 9)] = (40, 1)
    assert "reservingOrReservedGroup of cell 9: group 40 (not the group its name maps to) != group 40" in H.diff(a, ghost)
    for bad in ([99, 0], [H.FREE, 0, 3, 5, 1, 2], [H.BAD_NODE, 6, H.BAD_NODE, 2]):
        with pytest.raises(ValueError):
            H.decode(bad)


def test_the_api_fuzz_reports_a_corrupted_hidden_item_by_name(emu_lib, oracle_lib, monkeypatch):
    """Two entries of one free list swapped on one side only (every result and cell state stays equal): the fuzz run
    fails at the first call and says which list and position differ."""
    import fuzz_api
    raw = hidden_state.raw

    def corrupted(lib, ctx):
        w = raw(lib, ctx)
        if lib is emu_lib:
            i = 0
            while w[i] == hidden_state.FREE and w[i + 3] < 2:
                i += 4 + w[i + 3]
            assert w[i] == hidden_state.FREE
            w[i + 4], w[i + 5] = w[i + 5], w[i + 4]
        return w

    monkeypatch.setattr(hidden_state, "raw", corrupted)
    d = fuzz_api.run_seed(emu_lib, oracle_lib, 1, 3)
    assert d is not None and "op 0" in d and "hidden state differs: freeCellList[chain " in d and "position 0" in d, d


# ---------------------------------------------------------------------------------------------- CPU tier: emulation


@pytest.mark.parametrize("name", sorted(TRACES))
def test_emu_hidden_state_on_trace(emu_lib, oracle_lib, name, monkeypatch):
    states = check_trace(emu_lib, oracle_lib, name, monkeypatch)
    assert any(k[0] == hidden_state.USED_PHYSICAL for s in states for k in s)  # the trace does allocate


def test_emu_hidden_state_with_preemption_c4(emu_lib, oracle_lib, monkeypatch):
    check_c4(emu_lib, oracle_lib, C4, monkeypatch)


def test_emu_hidden_state_with_lazy_preemption(emu_lib, oracle_lib, monkeypatch):
    stats = check_c4(emu_lib, oracle_lib, C4_LAZY, monkeypatch)
    assert stats["lazy_preempted_groups"] > 0


def test_simt_hidden_state_on_small_c3_with_several_ctas(simt_lib, oracle_lib, monkeypatch):
    """The order in which the CTAs of a VC-parallel batch enter their shared sections decides the order of the free
    lists; the SIMT emulation runs small C3 (two VCs) on two CTAs."""
    t = small_c3(1000)
    ctas = []
    record = record_states(monkeypatch, ctas=ctas)
    ha, _, sa = run_trace(simt_lib, t, chunks=2)
    monkeypatch.undo()
    hb, sb, want = trace_states(oracle_lib, t, monkeypatch, chunks=2)
    assert ha == hb and sa == sb
    assert_same_states(record, want)
    assert max(ctas) > 1, ctas


def doomed_overflow_seen(oracle_lib, monkeypatch):
    """Wraps hidden_state.full to note, on the oracle's side, every doomed-bad list longer than the VC's preassigned
    cells of its (chain, level); returns the list of (vc, chain, level, length, preassigned) it appends to."""
    import ctypes as C
    seen, full = [], hidden_state.full

    def spy(lib, ctx, *names):
        s = full(lib, ctx, *names)
        if lib is oracle_lib:
            for k, v in s.items():
                if k[0] == hidden_state.DOOMED_BAD:
                    n = C.c_int32()
                    assert lib.hived_vc_preassigned_cells(ctx, k[1], k[2], k[3], None, 0, C.byref(n)) == 0
                    if len(v) > n.value:
                        seen.append(k[1:] + (len(v), n.value))
        return s

    monkeypatch.setattr(hidden_state, "full", spy)
    return seen


def test_doomed_bad_list_outgrows_the_preassigned_cells(emu_lib, oracle_lib, monkeypatch):
    """Synthetic-cluster fuzz seed 2098 (names re-used, Filtering-phase calls): a doomed bad cell whose leaves a pod used
    is unbound when the pod leaves but stays on the VC's doomed-bad list, its virtual cell is bound to the next bad
    cell, and at op 211 (setBadNode) the list holds more cells than the VC has preassigned cells at that level.  The
    device's segment used to be exactly that large and reported the overflow as the reference's panic."""
    seen = doomed_overflow_seen(oracle_lib, monkeypatch)
    assert run_fuzz_seed(emu_lib, oracle_lib, 2098, monkeypatch, **SYNTHETIC_NO_RENAME_FILTERING) is None
    assert seen, "the doomed-bad list no longer outgrows the preassigned cells in this seed"


def test_an_erased_ghost_keeps_its_id_while_cells_name_it(emu_lib, oracle_lib, monkeypatch):
    """Synthetic-cluster fuzz seed 365 (names re-used, Filtering-phase calls): a ghost group record that was itself
    erased by name (Core::eraseGroupByName) is still named by a cell.  hived_get_group reported such an id as not
    `referenced`, the mirror handed it back, and the cell's group became a different name on the device than in the
    oracle — visible only in the hidden state (usingGroup) until a later erase through that cell."""
    assert run_fuzz_seed(emu_lib, oracle_lib, 365, monkeypatch, **SYNTHETIC_NO_RENAME_FILTERING) is None


@pytest.mark.parametrize("seed", [782, 2385])
def test_emu_hidden_state_on_fuzz_seeds_of_the_other_anomalies(emu_lib, oracle_lib, seed, monkeypatch):
    """782: a free list holding one cell 16 times (Filtering-phase calls); 2385: a ghost group reached through a
    Reserved cell — both compared item by item after every call."""
    env = {"FUZZ_FILTERING": "1"} if seed == 782 else {}
    assert run_fuzz_seed(emu_lib, oracle_lib, seed, monkeypatch, **env) is None


def test_hooks_agree_on_a_fresh_cluster_and_honour_cap(emu_lib, oracle_lib):
    import ctypes as C
    words = []
    for lib in (emu_lib, oracle_lib):
        ctx = C.c_void_p()
        assert lib.hived_create(config.to_spec_text(config.config_c1()).encode(), None, C.byref(ctx)) == 0
        for n in range(lib.hived_num_nodes(ctx)):
            assert lib.hived_set_node_health(ctx, n, 1 if n % 3 else 0) == 0
        w = hidden_state.raw(lib, ctx)
        buf = (C.c_int32 * (len(w) + 4))(*([-7] * (len(w) + 4)))
        assert lib.hived_debug_state(ctx, buf, 5) == len(w)
        assert list(buf[:5]) == w[:5] and set(buf[5:]) == {-7}
        words.append(w)
        lib.hived_destroy(ctx)
    assert hidden_state.diff(*(hidden_state.decode(w) for w in words)) is None
    s = hidden_state.decode(words[0])
    # a third of C1's nodes bad: more bad cells than the VCs can spare, some are doomed
    assert {k[0] for k in s} >= {hidden_state.DOOMED_BAD, hidden_state.ALL_VC_DOOMED, hidden_state.BAD_NODE}


# ------------------------------------------------------------------------------------------------- GPU tier: CUDA


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(TRACES))
def test_cuda_hidden_state_on_trace(cuda_lib, oracle_lib, name, monkeypatch):
    """Through the batch kernel (VC-parallel where the batch allows it, then the repair kernel)."""
    check_trace(cuda_lib, oracle_lib, name, monkeypatch)


@pytest.mark.gpu
def test_cuda_hidden_state_with_preemption_c4(cuda_lib, oracle_lib, monkeypatch):
    check_c4(cuda_lib, oracle_lib, C4, monkeypatch)


@pytest.mark.gpu
def test_cuda_hidden_state_with_lazy_preemption(cuda_lib, oracle_lib, monkeypatch):
    assert check_c4(cuda_lib, oracle_lib, C4_LAZY, monkeypatch)["lazy_preempted_groups"] > 0


@pytest.mark.gpu
def test_cuda_hidden_state_on_small_c3_for_every_cta_count(cuda_lib, oracle_lib, monkeypatch, tmp_path):
    """Small C3 at HIVED_NCTA = 1, 2 and 16 (each in its own process: the CTA count is fixed when a context is
    created): the hidden state after every chunk — after the repair kernel — equals the oracle's."""
    _, _, want = trace_states(oracle_lib, TRACES["C3-small"](), monkeypatch)
    code = ("import pickle, sys; sys.path.insert(0, %r); sys.path.insert(0, %r)\n"
            "import pytest, test_hidden_state as T\n"
            "from hivedscheduler_b200 import _cabi\n"
            "mp = pytest.MonkeyPatch()\n"
            "_, _, s = T.trace_states(_cabi.load_cuda_library(), T.TRACES['C3-small'](), mp)\n"
            "pickle.dump(s, open(sys.argv[1], 'wb'))\n") % (os.path.dirname(HERE), HERE)
    for ncta in ("1", "2", "16"):
        out = tmp_path / ("states_%s.pkl" % ncta)
        subprocess.check_call([sys.executable, "-c", code, str(out)], env=dict(os.environ, HIVED_NCTA=ncta))
        with open(out, "rb") as f:
            got = pickle.load(f)
        try:
            assert_same_states(got, want)
        except AssertionError as e:
            raise AssertionError("HIVED_NCTA=%s: %s" % (ncta, e))


@pytest.mark.gpu
@pytest.mark.parametrize("seed,env", [(2098, SYNTHETIC_NO_RENAME_FILTERING), (365, SYNTHETIC_NO_RENAME_FILTERING),
                                      (782, {"FUZZ_FILTERING": "1"}), (2385, {})],
                         ids=["2098-synthetic", "365-synthetic", "782-filtering", "2385"])
def test_cuda_hidden_state_on_fuzz_seeds(cuda_lib, oracle_lib, seed, env, monkeypatch):
    """The per-call path (resident kernel): the API fuzz compares the hidden state after every call."""
    seen = doomed_overflow_seen(oracle_lib, monkeypatch) if seed == 2098 else None
    assert run_fuzz_seed(cuda_lib, oracle_lib, seed, monkeypatch, **env) is None
    if seen is not None:
        assert seen
