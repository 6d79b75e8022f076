"""CPU: the C-ABI library loads and exports every symbol include/snk.h declares; the host-only
entry points (layout, byte model, argument validation) agree with the oracle.  No GPU work."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import c_oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def L():
    import __graft_entry__ as ge
    if not os.path.exists(ge.LIB):
        ge.build()
    from snakes_b200 import _lib
    return _lib


def test_header_symbols_are_exported(L):
    header = open(os.path.join(ROOT, "include", "snk.h")).read()
    declared = set(re.findall(r"^\s*(?:int|const char\*)\s+(snk_\w+)\s*\(", header, flags=re.M))
    assert len(declared) >= 20
    lib = C.CDLL(L.LIB_PATH)
    for name in sorted(declared):
        assert hasattr(lib, name), "libsnk.so does not export %s" % name
    assert declared <= set(L._SIGNATURES), "python binding misses %s" % (declared - set(L._SIGNATURES))
    assert lib.snk_version() == int(re.search(r"#define SNK_VERSION (\d+)", header).group(1))


def test_no_torch_types_in_abi():
    header = open(os.path.join(ROOT, "include", "snk.h")).read()
    assert "torch" not in header.replace("no torch", "") and "at::" not in header and "#include <cuda" not in header


@pytest.mark.parametrize("rules,S,D,F,N", [("classic", 2, 19, 2, 1000), ("adversarial", 3, 10, 3, 17), ("cut", 16, 64, 16, 5)])
def test_state_layout_matches_oracle(L, rules, S, D, F, N):
    cfg = L.make_config(N, D, S, F, None, rules)
    lay = L.SnkStateLayout()
    L.check(L.lib().snk_state_layout_of(C.byref(cfg), C.byref(lay)))
    ocfg = c_oracle.make_config(N, size=D, n_snakes=S, n_fruits=F, rules=rules)
    olay = c_oracle.Layout()
    assert c_oracle.lib().so_state_layout_of(C.byref(ocfg), C.byref(olay)) == 0
    for name, _ in lay._fields_:
        assert getattr(lay, name) == getattr(olay, name), name
    assert lay.cap >= D * D + 1


def test_algorithmic_bytes_formula(L):
    # SURVEY.md section 8d: K*V^2*3 + 19S + 2*SigmaL + 2F + 30; configs[3] with SigmaL = 6 -> 2730
    cfg = L.make_config(131072, 19, 2, 2, 2, "classic")
    out = C.c_double(0)
    L.check(L.lib().snk_algorithmic_bytes_per_step(C.byref(cfg), 6.0, C.byref(out)))
    assert out.value == 2 * 21 * 21 * 3 + 19 * 2 + 2 * 6 + 2 * 2 + 30 == 2730


def test_bad_arguments_are_reported_not_crashed(L):
    lib = L.lib()
    lay = L.SnkStateLayout()
    bad = L.make_config(4, 1, 2)
    assert lib.snk_state_layout_of(C.byref(bad), C.byref(lay)) == -1
    assert b"size" in lib.snk_last_error()
    assert lib.snk_step(None, None, None) == -1
    assert lib.snk_destroy(None) == 0
    out = C.c_void_p()
    too_many = L.make_config(4, 10, 64)
    assert lib.snk_create(C.byref(too_many), C.byref(out)) == -1 and not out.value
    # header and cfg_check agree: n_fruits 0..32, env_id_base >= 0, global ids within 32 bits (ADVICE round 1)
    assert lib.snk_state_layout_of(C.byref(L.make_config(4, 10, 2, 32)), C.byref(lay)) == 0
    assert lib.snk_state_layout_of(C.byref(L.make_config(4, 10, 2, 33)), C.byref(lay)) == -1
    assert lib.snk_state_layout_of(C.byref(L.make_config(4, 10, 2, env_id_base=-2)), C.byref(lay)) == -1
    assert b"env_id_base" in lib.snk_last_error()
    assert lib.snk_state_layout_of(C.byref(L.make_config(4, 10, 2, env_id_base=(1 << 32) - 3)), C.byref(lay)) == -1
    assert "0..32" in open(os.path.join(ROOT, "include", "snk.h")).read()
    # the entry points added in round 2 validate their arguments too
    assert lib.snk_graph_create(None, None, 1, 1, None, None, None, 0, None) == -1
    assert lib.snk_graph_launch(None, None) == -1 and lib.snk_graph_destroy(None) == 0
    assert lib.snk_comm_init(None, None, 1, 0) == -1 and lib.snk_comm_unique_id(None) == -1
    assert lib.snk_host_alloc(None, 16, None, None) == -1 and lib.snk_dump_state_range(None, 0, 1, None, 0) == -1
    assert set(L.DEVERR) == {1, 2, 4, 8, 16}
    # the debug string: an unknown key or an unlisted value is rejected by name before any CUDA call
    ok_cfg = L.make_config(4, 10, 2)
    for opts in (b"store=stg", b"paint2=0", b"lane=bogus", b"lane=split,restor_thr=1"):
        out = C.c_void_p()
        assert lib.snk_create_ex(C.byref(ok_cfg), opts, C.byref(out)) == -1 and not out.value
        assert opts.split(b",")[-1] in lib.snk_last_error()
    # an empty string and known keys get past that check (without a GPU, creation then fails with SNK_ECUDA)
    for opts in (b"", b"lane=split,restore_thr=2,epw=8"):
        out = C.c_void_p()
        rc = lib.snk_create_ex(C.byref(ok_cfg), opts, C.byref(out))
        assert rc in (0, -2), (opts, rc, lib.snk_last_error())
        if rc == 0:
            lib.snk_destroy(out)


def test_product_does_not_import_oracle():
    """The shipped package must never route through the CPU oracle."""
    pkg = os.path.join(ROOT, "snakes_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert "snake_oracle" not in src and "c_oracle" not in src and "libsnake_oracle" not in src, f
