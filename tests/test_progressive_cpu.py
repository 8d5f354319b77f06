"""CPU-only checks of the progressive-rendering ABI (vrj_render_progressive): the ctypes and Rust mirrors of its structs."""
import ctypes as C
import os
import re
import subprocess

from vanrijn_b200 import capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PAIRS = [("VrjProgressiveParams", capi.ProgressiveParams), ("VrjProgressiveStats", capi.ProgressiveStats)]


def test_progressive_struct_layouts_match_the_header(tmp_path):
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
    assert int(got["VrjProgressiveParams"]) == 32 and int(got["VrjProgressiveStats"]) == 40
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


def test_rust_default_params_are_valid():
    crate = open(os.path.join(ROOT, "rust", "vanrijn-cuda-sys", "src", "lib.rs")).read()
    m = re.search(r"VrjProgressiveParams \{ min_samples: (\d+), max_samples: (\d+), pass_samples: (\d+), max_passes: (\d+), "
                  r"rel_error: ([\d.e-]+), abs_floor: ([\d.e-]+) \}", crate)
    mn, mx, ps, mp = (int(x) for x in m.groups()[:4])
    rel, floor = float(m.group(5)), float(m.group(6))
    assert mn >= 2 and mx >= mn and ps >= 1 and rel > 0 and floor >= 0
