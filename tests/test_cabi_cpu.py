"""CPU tests (-m "not gpu") of the boundary: the C-ABI library builds, loads, exports every symbol
include/polars_b200.h declares, and fails loudly (no CPU fallback) when no GPU is present."""
import ctypes as C
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    src = open(os.path.join(ROOT, "include", "polars_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(bl_[a-z0-9_]+)\s*\(", src)))


def test_header_declares_the_hot_path():
    syms = declared_symbols()
    for s in ("bl_elementwise", "bl_compare", "bl_filter", "bl_filter_cmp", "bl_gather", "bl_groupby_agg", "bl_groupby_agg_keys", "bl_group_tuples", "bl_hash_join", "bl_join",
              "bl_hash_partition", "bl_groupby_create", "bl_groupby_consume", "bl_groupby_export_partials",
              "bl_groupby_merge_partials", "bl_groupby_finish", "bl_last_error", "bl_init", "bl_alloc_pinned"):
        assert s in syms


def test_library_exports_every_declared_symbol():
    import polars_b200 as plb
    lib = plb.lib()
    missing = [s for s in declared_symbols() if not hasattr(lib, s)]
    assert not missing, f"declared in include/polars_b200.h but not exported: {missing}"
    assert lib.bl_abi_version() == 1


def test_plugin_abi_symbols_exported():
    # boundary B1 (crates/polars-plan/src/plans/aexpr/function_expr/plugin.rs:70-217)
    import polars_b200 as plb
    lib = plb.lib()
    lib._polars_plugin_get_version.restype = C.c_uint32
    assert lib._polars_plugin_get_version() == (0 << 16) + 1          # polars-ffi/src/lib.rs:12-17
    for op in ("add", "sub", "mul", "floordiv", "mod", "truediv", "eq", "ne", "lt", "le", "gt", "ge", "filter", "gather",
               "group_sum", "group_mean", "group_min", "group_max", "group_count", "join_inner_idx"):
        assert hasattr(lib, f"_polars_plugin_bl_{op}"), op
        assert hasattr(lib, f"_polars_plugin_field_bl_{op}"), op
    assert hasattr(lib, "_polars_plugin_get_last_error_message")


def test_no_gpu_fails_loudly_no_cpu_fallback():
    import torch
    if torch.cuda.device_count():      # any visible device, whatever its /dev node is called
        pytest.skip("needs a machine without a GPU")
    import polars_b200 as plb
    with pytest.raises(plb.B200Error) as e:
        plb.elementwise("add", np.arange(4), np.arange(4))
    assert "no CPU fallback" in str(e.value) and e.value.status == 2
    with pytest.raises(plb.B200Error):
        plb.group_by_agg(np.arange(4), [("len", None)])


def test_product_never_imports_the_oracle():
    for dirpath, _, files in os.walk(os.path.join(ROOT, "polars_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp")):
                txt = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(import|from)\s+oracle\b", txt, flags=re.M), f
                assert "liboracle" not in txt and "oracle.c" not in txt and "or_group_by" not in txt, f


def _build_c_demo(tmp_path):
    import shutil
    import subprocess
    cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else shutil.which("gcc")
    if cc is None:
        pytest.skip("no C compiler")
    import polars_b200 as plb
    plb.lib()                                     # builds the library if needed
    libdir = os.path.join(ROOT, "polars_b200", "_lib")
    exe = str(tmp_path / "c_abi_demo")
    r = subprocess.run([cc, "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I" + os.path.join(ROOT, "include"), os.path.join(ROOT, "examples", "c_abi_demo.c"),
                        "-L" + libdir, "-lpolars_b200", "-Wl,-rpath," + libdir, "-o", exe], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return exe


def test_header_is_plain_c_and_links(tmp_path):
    # the boundary must be consumable from C99 (no C++ / torch types): compile + link examples/c_abi_demo.c
    _build_c_demo(tmp_path)


def test_rust_sys_declarations_match_the_header():
    # integration/polars_b200_sys.rs (boundary B3, documentation: no Rust toolchain here) is generated from the header;
    # it must declare every exported entry point with the header's current signature
    import subprocess
    import sys
    r = subprocess.run([sys.executable, os.path.join(ROOT, "integration", "gen_rust_sys.py"), "--check"])
    assert r.returncode == 0, "integration/polars_b200_sys.rs is stale: run python integration/gen_rust_sys.py"
    rs = open(os.path.join(ROOT, "integration", "polars_b200_sys.rs")).read()
    for sym in declared_symbols():
        assert f"pub fn {sym}(" in rs, sym
