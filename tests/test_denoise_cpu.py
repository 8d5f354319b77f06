"""CPU-only checks of the denoiser ABI (vrj_render_aux, vrj_denoise): the ctypes and Rust mirrors of its structs, and the
default parameters stated in the header, host.py and the Rust crate."""
import ctypes as C
import os
import re
import subprocess

from vanrijn_b200 import capi, host

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PAIRS = [("VrjAuxOut", capi.AuxOut), ("VrjDenoiseParams", capi.DenoiseParams)]


def header():
    return open(os.path.join(ROOT, "include", "vanrijn_cuda.h")).read()


def crate():
    return open(os.path.join(ROOT, "rust", "vanrijn-cuda-sys", "src", "lib.rs")).read()


def test_denoise_struct_layouts_match_the_header(tmp_path):
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
    assert int(got["VrjAuxOut"]) == 48 and int(got["VrjDenoiseParams"]) == 32
    for cname, ct in PAIRS:
        assert int(got[cname]) == C.sizeof(ct), cname
        for fname, _ in ct._fields_:
            assert int(got["%s.%s" % (cname, fname)]) == getattr(ct, fname).offset, (cname, fname)


def c_fields(name):
    """Field names of a header struct in order, declarations with several names (`uint32_t memory, pad;`) and pointers included."""
    body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (name, name), header(), re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = []
    for decl in body.split(";"):
        decl = decl.strip()
        if not decl:
            continue
        m = re.match(r"(?:const\s+)?\w+\s+(.*)", decl, re.S)
        names += [part.strip().lstrip("*").strip() for part in m.group(1).split(",")]
    return names


def test_rust_mirrors_list_the_header_fields_in_order():
    for name, ct in PAIRS:
        r_body = re.search(r"pub struct %s \{(.*?)\}" % name, crate(), re.S).group(1)
        assert re.findall(r"pub (\w+):", r_body) == c_fields(name) == [f for f, _ in ct._fields_], name


def test_default_parameters_agree():
    h = header()
    d = {k: float(re.search(r"#define VRJ_DENOISE_DEFAULT_%s (\S+)" % k, h).group(1))
         for k in ("ITERATIONS", "SIGMA_LUMINANCE", "SIGMA_NORMAL", "SIGMA_DEPTH")}
    assert (host.DENOISE_ITERATIONS, host.DENOISE_SIGMA_LUMINANCE, host.DENOISE_SIGMA_NORMAL, host.DENOISE_SIGMA_DEPTH) == \
        (d["ITERATIONS"], d["SIGMA_LUMINANCE"], d["SIGMA_NORMAL"], d["SIGMA_DEPTH"])
    m = re.search(r"VrjDenoiseParams \{ iterations: (\d+), pad: 0, sigma_luminance: ([\d.e-]+), sigma_normal: ([\d.e-]+), "
                  r"sigma_depth: ([\d.e-]+) \}", crate())
    assert tuple(float(x) for x in m.groups()) == (d["ITERATIONS"], d["SIGMA_LUMINANCE"], d["SIGMA_NORMAL"], d["SIGMA_DEPTH"])
