"""CPU: the C-ABI library loads and exports every symbol include/betazero_b200.h declares; the
ctypes mirror structs have the layout of the C structs.  No compute calls (no GPU here)."""
import ctypes as C
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "betazero_b200.h")


def _declared_functions():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(?:int|int64_t|const char \*)\s*(bz_[a-z0-9_]+)\s*\(", src)))


def test_header_symbols_are_exported_and_bound():
    from betazero_b200 import _lib

    names = _declared_functions()
    assert len(names) >= 20
    lib = _lib.load()
    for n in names:
        assert hasattr(lib, n), f"{n} declared in the header but not exported"
    assert sorted(_lib.SIGNATURES) == names, "ctypes table and header disagree"
    assert lib.bz_abi_version() == _lib.ABI_VERSION == 6
    assert lib.bz_error_string(0) == b"ok" and b"argument" in lib.bz_error_string(-1)


def test_no_unexpected_dependencies():
    """the boundary is a plain C ABI: no libtorch / libpython in the link line"""
    from betazero_b200 import _lib

    out = subprocess.run(["ldd", _lib.lib_path()], capture_output=True, text=True).stdout
    assert "libtorch" not in out and "libpython" not in out and "libc10" not in out


def test_struct_layouts_match_the_c_compiler(tmp_path):
    """compile a tiny C program against the header and compare sizeof/offsetof with ctypes"""
    from betazero_b200._lib import BzSelfplayState, BzTreePools

    fields_p = [n for n, _ in BzTreePools._fields_]
    fields_s = [n for n, _ in BzSelfplayState._fields_]
    prog = ['#include <stdio.h>', '#include <stddef.h>', f'#include "{HEADER}"', "int main(void){",
            'printf("%zu\\n", sizeof(bz_tree_pools));']
    prog += [f'printf("%zu\\n", offsetof(bz_tree_pools, {f}));' for f in fields_p]
    prog += ['printf("%zu\\n", sizeof(bz_selfplay_state));']
    prog += [f'printf("%zu\\n", offsetof(bz_selfplay_state, {f}));' for f in fields_s]
    prog += ["return 0;}"]
    src = tmp_path / "layout.c"
    src.write_text("\n".join(prog))
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-o", str(exe), str(src)])
    vals = [int(v) for v in subprocess.check_output([str(exe)], text=True).split()]
    exp = [C.sizeof(BzTreePools)] + [getattr(BzTreePools, f).offset for f in fields_p]
    exp += [C.sizeof(BzSelfplayState)] + [getattr(BzSelfplayState, f).offset for f in fields_s]
    assert vals == exp


def test_compute_path_refuses_cpu_tensors():
    """there is no CPU fallback: handing the engine a host tensor is an error, not a slow path"""
    import torch

    from betazero_b200 import _lib

    with pytest.raises(_lib.BzError, match="CUDA tensor"):
        _lib.dptr(torch.zeros(4, dtype=torch.int64))


def test_product_never_imports_the_oracle():
    """the oracle is test infrastructure: nothing under betazero_b200/ may import, load or link it"""
    pkg = os.path.join(ROOT, "betazero_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if not f.endswith((".py", ".cu", ".cuh", ".h")):
                continue
            txt = open(os.path.join(dirpath, f)).read()
            assert "liboracle" not in txt and "pyoracle" not in txt, f"{f} references the oracle library"
            assert not re.search(r"^\s*(from|import)\s+oracle\b", txt, flags=re.M), f"{f} imports the oracle"
            assert not re.search(r"#include\s+[\"<].*oracle", txt), f"{f} includes oracle code"


def test_abi_version_has_one_source_of_truth():
    """the header, the ctypes mirror and the driver's build() check must agree (build() once asserted a literal)"""
    import re

    from betazero_b200 import _lib

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    header = open(os.path.join(root, "include", "betazero_b200.h")).read()
    assert int(re.search(r"#define BZ_ABI_VERSION (\d+)", header).group(1)) == _lib.ABI_VERSION
    entry = open(os.path.join(root, "__graft_entry__.py")).read()
    assert "bz_abi_version() == _lib.ABI_VERSION" in entry


def test_library_staleness_is_decided_by_content_not_by_file_times():
    """a snapshot copied to the GPU box does not keep mtimes; a rebuild there, started by every rank of a torchrun job
    at once, once produced 'file too short' on dlopen"""
    from betazero_b200 import build as bz_build

    bz_build.build()
    assert not bz_build.needs_build()
    src = os.path.join(bz_build.CSRC, "env.cu")
    st = os.stat(src)
    try:
        os.utime(src, None)  # newer than the library
        assert not bz_build.needs_build()
    finally:
        os.utime(src, (st.st_atime, st.st_mtime))


def test_concurrent_oracle_builds_do_not_race():
    """four processes find the oracle library stale at the same time: one builds under the lock, all of them load a
    complete library"""
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    stamp = os.path.join(root, "oracle", "liboracle.so.srchash")
    if os.path.exists(stamp):
        os.remove(stamp)
    code = ("import sys; sys.path.insert(0, %r); from oracle import pyoracle as po; "
            "import numpy as np; m = po.legal_mask(np.array([0x0000000810000000], np.uint64), np.array([0x0000001008000000], np.uint64)); "
            "print(int(m[0]))" % root)
    procs = [subprocess.Popen([sys.executable, "-c", code], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True) for _ in range(4)]
    outs = [p.communicate(timeout=300) for p in procs]
    assert all(p.returncode == 0 for p in procs), [o[1][-500:] for o in outs]
    assert len({o[0].strip() for o in outs}) == 1 and os.path.exists(stamp)
