"""CPU-only checks of the adaptive-sampling ABI (vrj_render_adaptive): the ctypes and Rust mirrors of its structs."""
import ctypes as C
import os
import re
import subprocess

from vanrijn_b200 import capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_adaptive_struct_layouts_match_the_header(tmp_path):
    pairs = [("VrjAdaptiveParams", capi.AdaptiveParams), ("VrjAdaptiveStats", capi.AdaptiveStats)]
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "vanrijn_cuda.h"', 'int main(void){']
    for cname, ct in pairs:
        lines.append('printf("%s %%zu\\n", sizeof(%s));' % (cname, cname))
        for fname, _ in ct._fields_:
            lines.append('printf("%s.%s %%zu\\n", offsetof(%s, %s));' % (cname, fname, cname, fname))
    lines.append('return 0;}')
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)], check=True)
    got = dict(l.split() for l in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines())
    assert int(got["VrjAdaptiveParams"]) == 32 and int(got["VrjAdaptiveStats"]) == 32
    for cname, ct in pairs:
        assert int(got[cname]) == C.sizeof(ct), cname
        for fname, _ in ct._fields_:
            assert int(got["%s.%s" % (cname, fname)]) == getattr(ct, fname).offset, (cname, fname)


def test_rust_mirrors_list_the_header_fields_in_order():
    header = open(os.path.join(ROOT, "include", "vanrijn_cuda.h")).read()
    crate = open(os.path.join(ROOT, "rust", "vanrijn-cuda-sys", "src", "lib.rs")).read()
    for name in ("VrjAdaptiveParams", "VrjAdaptiveStats"):
        body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (name, name), header, re.S).group(1)
        c_fields = re.findall(r"\b(?:uint32_t|uint64_t|double)\s+(\w+);", body)
        r_body = re.search(r"pub struct %s \{(.*?)\}" % name, crate, re.S).group(1)
        assert re.findall(r"pub (\w+):", r_body) == c_fields, name
