"""CPU-only checks of the count-map ABI (vrj_render_counts, vrj_plan_counts): the ctypes and Rust mirrors of its structs,
and the function declarations of the mirrors."""
import ctypes as C
import os
import re
import subprocess

from vanrijn_b200 import capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PAIRS = [("VrjCountsStats", capi.CountsStats), ("VrjPlanStats", capi.PlanStats)]


def test_counts_struct_layouts_match_the_header(tmp_path):
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "vanrijn_cuda.h"', 'int main(void){']
    for cname, ct in PAIRS:
        lines.append('printf("%s %%zu\\n", sizeof(%s));' % (cname, cname))
        for fname, _ in ct._fields_:
            lines.append('printf("%s.%s %%zu\\n", offsetof(%s, %s));' % (cname, fname, cname, fname))
    lines.append('return 0;}')
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)], check=True)
    got = dict(l.split() for l in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines())
    assert int(got["VrjCountsStats"]) == 24 and int(got["VrjPlanStats"]) == 32
    for cname, ct in PAIRS:
        assert int(got[cname]) == C.sizeof(ct), cname
        for fname, _ in ct._fields_:
            assert int(got["%s.%s" % (cname, fname)]) == getattr(ct, fname).offset, (cname, fname)


def test_rust_mirrors_list_the_header_fields_in_order():
    header = open(os.path.join(ROOT, "include", "vanrijn_cuda.h")).read()
    crate = open(os.path.join(ROOT, "rust", "vanrijn-cuda-sys", "src", "lib.rs")).read()
    for name, ct in PAIRS:
        body = re.sub(r"/\*.*?\*/", "", re.search(r"typedef struct %s \{(.*?)\} %s;" % (name, name), header, re.S).group(1), flags=re.S)
        c_fields = [f.strip() for decl in re.findall(r"\b(?:uint32_t|uint64_t|double)\s+([\w\s,]+);", body) for f in decl.split(",")]
        r_body = re.search(r"pub struct %s \{(.*?)\}" % name, crate, re.S).group(1)
        assert re.findall(r"pub (\w+):", r_body) == c_fields == [f for f, _ in ct._fields_], name
        assert all(t == "u64" for t in re.findall(r"pub \w+: (\w+)", r_body)), name


def _params(decl):
    """the parameter names of a C or Rust declaration, in order"""
    inner = decl[decl.index("(") + 1:decl.rindex(")")]
    return [re.findall(r"(\w+)\s*$", p.split(":")[0].strip())[0] for p in inner.split(",")]


def test_declarations_agree_across_the_header_rust_and_ctypes():
    header = re.sub(r"\s+", " ", open(os.path.join(ROOT, "include", "vanrijn_cuda.h")).read())
    crate = re.sub(r"\s+", " ", open(os.path.join(ROOT, "rust", "vanrijn-cuda-sys", "src", "lib.rs")).read())
    for fn, n in (("vrj_render_counts", 9), ("vrj_plan_counts", 9)):
        c = re.search(r"VRJ_API VrjStatus %s\(([^)]*)\);" % fn, header).group(0)
        r = re.search(r"pub fn %s\(([^)]*)\) -> i32;" % fn, crate).group(0)
        assert _params(c) == _params(r) and len(_params(c)) == n, fn
        assert fn in capi.CUDA_SYMBOLS
    # the argtypes the ctypes loader declares have one entry per parameter
    src = open(os.path.join(ROOT, "vanrijn_b200", "capi.py")).read()
    for fn in ("vrj_render_counts", "vrj_plan_counts"):
        assert "L.%s.argtypes" % fn in src and "L.%s.restype = C.c_int32" % fn in src
