"""The product library loads and exports every symbol include/hived.h declares (no compute without a GPU)."""
import ctypes as C
import os
import re

import pytest

from hivedscheduler_b200 import _cabi, config

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols(header="hived.h"):
    src = open(os.path.join(ROOT, "include", header)).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(hived_[a-z_0-9]+)\s*\(", src)))


def test_header_symbols_are_bound_and_exported():
    import __graft_entry__ as g
    g.build_cuda()
    lib = _cabi.load_cuda_library()
    bound = {name for name, _, _ in _cabi.SYMBOLS}
    for sym in declared_symbols():
        assert sym in bound, "include/hived.h declares %s but _cabi does not bind it" % sym
        assert getattr(lib, sym) is not None
    assert lib.hived_backend() == b"cuda-sm100a"
    # the other headers of include/: measurement hooks, multi-GPU partition, request ingest
    from hivedscheduler_b200 import dist, frontend, ingest
    dist.bind_multigpu(lib)
    ingest.bind(lib)
    frontend.bind(lib)
    typed = {n for n, _, _ in ingest.SYMBOLS} | {n for n, _, _ in frontend.SYMBOLS}
    for header in ("hived_bench.h", "hived_multigpu.h", "hived_ingest.h", "hived_frontend.h"):
        syms = declared_symbols(header)
        assert syms, header
        for sym in syms:
            assert getattr(lib, sym) is not None, "%s declares %s but the library does not export it" % (header, sym)
            if header in ("hived_ingest.h", "hived_frontend.h"):
                assert sym in typed, sym


def test_struct_layouts_match_header():
    # sizes the C compiler computes for the structs of include/hived.h
    import subprocess, tempfile
    prog = r'''
#include <stdio.h>
#include "hived.h"
int main(){printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu %zu\n",sizeof(hived_options_t),sizeof(hived_pod_spec_t),sizeof(hived_result_t),
sizeof(hived_bind_info_t),sizeof(hived_event_t),sizeof(hived_group_info_t),sizeof(hived_cell_status_t),sizeof(hived_stats_t),
sizeof(hived_group_placement_t),sizeof(hived_cell_info_t));return 0;}
'''
    with tempfile.TemporaryDirectory() as d:
        open(os.path.join(d, "a.c"), "w").write(prog)
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), "-o", os.path.join(d, "a"), os.path.join(d, "a.c")])
        sizes = [int(x) for x in subprocess.check_output([os.path.join(d, "a")]).split()]
    assert sizes == [C.sizeof(x) for x in (_cabi.Options, _cabi.PodSpec, _cabi.Result, _cabi.BindInfo, _cabi.Event,
                                           _cabi.GroupInfo, _cabi.CellStatus, _cabi.Stats, _cabi.GroupPlacement,
                                           _cabi.CellInfo)]


def test_product_fails_loudly_without_a_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    lib = _cabi.load_cuda_library()
    ctx = C.c_void_p()
    rc = lib.hived_create(config.to_spec_text(config.config_c1()).encode(), None, C.byref(ctx))
    assert rc == 103  # HIVED_ERR_NO_DEVICE: there is no CPU fallback
    assert b"no CPU fallback" in lib.hived_create_error()


def test_missing_extension_is_an_error(tmp_path):
    with pytest.raises(_cabi.MissingExtension):
        _cabi.load_library(str(tmp_path / "libhived_cuda.so"))


def test_state_hooks_are_declared_and_exported_by_every_implementation(emu_lib, oracle_lib):
    """hived_debug_view_hash / hived_debug_state are test hooks of include/hived_bench.h: the product exports them
    (test_header_symbols_are_bound_and_exported) and so do the implementations the tests compare it with; the section
    tags of the encoding are the ones tests/hidden_state.py decodes."""
    import hidden_state
    assert {"hived_debug_view_hash", "hived_debug_state"} <= set(declared_symbols("hived_bench.h"))
    for lib in (emu_lib, oracle_lib):
        assert getattr(lib, "hived_debug_view_hash") is not None and getattr(lib, "hived_debug_state") is not None
    src = open(os.path.join(ROOT, "include", "hived_bench.h")).read()
    tags = {m[0]: int(m[1]) for m in re.findall(r"HIVED_DS_([A-Z_]+)\s*=\s*(\d+)", src)}
    assert tags and tags == {k: getattr(hidden_state, k) for k in tags}
