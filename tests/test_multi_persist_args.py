"""The multi-shard persistence and read-back entry points without a GPU: NULL arguments are refused before any device
work, every new dawn_multi_* name is declared in include/dawn_index.h and exported by the library, and the Rust
MultiIndex offers the methods search_provider.rs calls on an Index."""
import ctypes as C
import os
import re
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEW = ["dawn_multi_save", "dawn_multi_load", "dawn_multi_get", "dawn_multi_get_i24", "dawn_multi_verify",
       "dawn_multi_search_i24"]
INVALID = -1


def test_null_handle_and_arguments_are_invalid(dawn):
    L = dawn.index.load_library()
    v = np.zeros(384, dtype=np.float32)
    w = np.zeros(1152, dtype=np.uint8)
    lab, dist, n = np.zeros(4, dtype=np.uint64), np.zeros(4, dtype=np.float32), C.c_size_t(7)
    bad, lo, hi = C.c_size_t(0), C.c_float(0), C.c_float(0)
    p = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    assert L.dawn_multi_save(None, b"/nonexistent/x") == INVALID
    assert L.dawn_multi_load(None, b"/nonexistent/x") == INVALID
    assert L.dawn_multi_get(None, 1, p(v)) == INVALID
    assert L.dawn_multi_get_i24(None, 1, p(w)) == INVALID
    assert L.dawn_multi_verify(None, C.byref(bad), C.byref(lo), C.byref(hi)) == INVALID
    assert L.dawn_multi_search_i24(None, p(w), 4, 0, 0.0, p(lab), p(dist), C.byref(n)) == INVALID
    assert "null" in L.dawn_multi_last_error().decode()


def _header_names():
    header = open(os.path.join(ROOT, "include", "dawn_index.h")).read()
    return set(re.findall(r"\b(dawn_[a-z0-9_]+)\s*\(", re.sub(r"/\*.*?\*/", "", header, flags=re.S)))


def test_new_names_are_declared_and_exported(dawn):
    assert set(NEW) <= _header_names()
    out = subprocess.run(["nm", "-D", "--defined-only", dawn.index.LIB_PATH], capture_output=True, text=True).stdout
    exported = set(re.findall(r" T (dawn_[a-z0-9_]+)", out))
    assert set(NEW) <= exported, set(NEW) - exported


def test_rust_multi_index_has_the_index_methods():
    shim = open(os.path.join(ROOT, "rust", "src", "index", "gpu_index.rs")).read()
    impl = re.search(r"impl MultiIndex \{(.*?)\n\}", shim, flags=re.S).group(1)
    index_impl = "".join(re.findall(r"impl Index \{(.*?)\n\}", shim, flags=re.S))
    for name in ("save", "load", "view", "get", "get_i24", "verify", "search_i24"):
        sig = re.search(rf"pub fn {name}\((.*?)\)\s*->\s*([^{{]+)\{{", impl)
        want = re.search(rf"pub fn {name}\((.*?)\)\s*->\s*([^{{]+)\{{", index_impl)
        assert sig and want, name
        assert sig.groups() == want.groups(), (name, sig.groups(), want.groups())
    block = re.search(r'extern "C" \{(.*?)\n\}', shim, flags=re.S).group(1)
    assert set(NEW) <= set(re.findall(r"fn (dawn_[a-z0-9_]+)\(", block))
