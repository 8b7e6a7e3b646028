"""The ctypes mirrors of the result and parameter structs (tokzig_b200.EncodeParams, BatchResult, CompactResult) against the C
compiler's layout of include/tokzig_b200.h: a small host probe prints sizeof / offsetof of every field."""
import ctypes as C
import os
import subprocess

import pytest

import tokzig_b200 as tz

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STRUCTS = (("tkz_encode_params", tz.EncodeParams), ("tkz_batch_result", tz.BatchResult), ("tkz_compact_result", tz.CompactResult))


@pytest.fixture(scope="module")
def layout(tmp_path_factory):
    d = tmp_path_factory.mktemp("abi")
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "tokzig_b200.h"', "int main(void) {"]
    for cname, py in STRUCTS:
        lines.append(f'    printf("{cname} sizeof %zu\\n", sizeof({cname}));')
        for f, _ in py._fields_:
            lines.append(f'    printf("{cname} {f} %zu\\n", offsetof({cname}, {f}));')
    lines += ["    return 0;", "}"]
    src, exe = d / "probe.c", d / "probe"
    src.write_text("\n".join(lines) + "\n")
    subprocess.check_call(["gcc", "-std=c11", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    out = {}
    for line in subprocess.check_output([str(exe)], text=True).splitlines():
        s, f, v = line.split()
        out[(s, f)] = int(v)
    return out


@pytest.mark.parametrize("cname,py", STRUCTS, ids=[s for s, _ in STRUCTS])
def test_ctypes_mirror_matches_the_header(layout, cname, py):
    assert C.sizeof(py) == layout[(cname, "sizeof")]
    for f, _ in py._fields_:
        assert getattr(py, f).offset == layout[(cname, f)], f


def test_overflow_fields_are_appended():
    assert [f for f, _ in tz.EncodeParams._fields_][-1] == "stride"
    assert [f for f, _ in tz.BatchResult._fields_][-3:] == ["n_rows", "row_tok_off", "doc_row_off"]
