"""spex_long_plan and spex_spmm_epilogue cross the C-ABI by value of their layout: the ctypes mirrors
(_capi.LongPlan, _capi.SpmmEpilogue) must list the header's fields in the same order with the same kinds, or every
plan / epilogue the library reads is garbage."""
import ctypes
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _assert_mirrors_header_struct(c_name, py_struct):
    hdr = open(os.path.join(ROOT, "include", "spex_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (c_name, c_name), hdr, flags=re.S).group(1)
    fields = re.findall(r"^\s*([A-Za-z_][\w\s*]*?)\s*\b(\w+);", body, flags=re.M)
    assert len(fields) == body.count(";"), "one field per declaration"

    def kind_c(t):
        t = " ".join(t.replace("*", " * ").split())
        if t.endswith("* const *"):
            return "pp"
        if "*" in t:
            return "p"
        return {"int32_t": "i32", "int64_t": "i64", "float": "f"}[t.replace("const", "").strip()]

    def kind_py(t):
        if t is ctypes.POINTER(ctypes.c_void_p):
            return "pp"
        return {ctypes.c_int32: "i32", ctypes.c_int64: "i64", ctypes.c_float: "f"}.get(t, "p")

    assert [(n, kind_c(t)) for t, n in fields] == [(n, kind_py(t)) for n, t in py_struct._fields_]


def test_long_plan_ctypes_matches_the_header_struct():
    from spex_b200 import _capi

    _assert_mirrors_header_struct("spex_long_plan", _capi.LongPlan)


def test_spmm_epilogue_ctypes_matches_the_header_struct():
    from spex_b200 import _capi

    _assert_mirrors_header_struct("spex_spmm_epilogue", _capi.SpmmEpilogue)
