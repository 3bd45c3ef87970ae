"""spex_long_plan crosses the C-ABI by value of its layout: the ctypes mirror (_capi.LongPlan) must list the
header's fields in the same order with the same kinds, or every plan the library reads is garbage."""
import ctypes
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_long_plan_ctypes_matches_the_header_struct():
    from spex_b200 import _capi

    hdr = open(os.path.join(ROOT, "include", "spex_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    body = re.search(r"typedef struct spex_long_plan \{(.*?)\} spex_long_plan;", hdr, flags=re.S).group(1)
    fields = re.findall(r"^\s*([A-Za-z_][\w\s]*?\**)\s*\b(\w+);", body, flags=re.M)

    def kind_c(t):
        if "*" in t:
            return "p"
        return {"int32_t": "i32", "int64_t": "i64"}[t.replace("const", "").strip()]

    def kind_py(t):
        return {ctypes.c_int32: "i32", ctypes.c_int64: "i64"}.get(t, "p")

    assert [(n, kind_c(t)) for t, n in fields] == [(n, kind_py(t)) for n, t in _capi.LongPlan._fields_]
