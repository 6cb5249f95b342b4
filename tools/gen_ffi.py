#!/usr/bin/env python3
"""Regenerates the `extern "C"` block of shim/src/ffi.rs from include/bpg.h (run after changing the header;
tests/test_abi_and_host.py::test_rust_ffi_matches_header fails until the two agree)."""
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE = {"int": "i32", "unsigned": "u32", "size_t": "usize", "uint8_t": "u8", "uint32_t": "u32", "uint64_t": "u64", "float": "f32", "double": "f64",
        "void": "c_void", "long": "i64", "bpg_ctx": "BpgCtx", "bpg_circuit": "BpgCircuit", "bpg_transcript": "BpgTranscript"}
RET = {"int": "i32", "void": None, "long": "i64", "size_t": "usize", "uint64_t": "u64", "const char *": "*const c_char", "bpg_transcript *": "*mut BpgTranscript"}


def param(p):
    p = p.strip()
    if p == "void":
        return None
    m = re.match(r"(.*?)([A-Za-z_][A-Za-z0-9_]*)(\[[0-9]*\](\[[0-9]*\])?)?$", p)
    ty, name, arr = m.group(1).strip(), m.group(2), m.group(3)
    if ty == "bpg_allgather_fn":
        return name, "Option<BpgAllgatherFn>"
    const = "const" in ty
    base = ty.replace("const", "").replace("*", "").strip()
    stars = ty.count("*") + (1 if arr else 0)
    if stars == 2 and const and base == "bpg_circuit":   # bpg_circuit *const *circuits
        return name, "*const *mut BpgCircuit"
    if stars == 2 and const and base == "uint8_t" and not ty.startswith("const"):  # uint8_t *const *proofs
        return name, "*const *mut u8"
    if stars == 2 and const and base == "uint8_t":       # const uint8_t *const *labels
        return name, "*const *const u8"
    rt = BASE[base]
    for i in range(stars):
        rt = ("*const " if const else "*mut ") + rt
    if stars == 2 and not const:
        rt = "*mut *mut " + BASE[base]
    return name, rt


def main():
    hdr = open(os.path.join(ROOT, "include", "bpg.h")).read()
    h = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    protos = re.findall(r"\n\s*([A-Za-z_][A-Za-z0-9_ \*]*?)\b(bpg_[a-z0-9_]+)\s*\(([^;]*?)\)\s*;", h)
    lines = []
    for ret, name, args in protos:
        ps = [param(a) for a in " ".join(args.split()).split(",")]
        ps = [p for p in ps if p]
        r = RET[ret.strip()]
        lines.append("    pub fn %s(%s)%s;" % (name, ", ".join("%s: %s" % p for p in ps), (" -> " + r) if r else ""))
    path = os.path.join(ROOT, "shim", "src", "ffi.rs")
    src = open(path).read()
    head, rest = src.split('extern "C" {\n', 1)
    tail = rest[rest.index("\n}\n"):]
    open(path, "w").write(head + 'extern "C" {\n' + "\n".join(lines) + tail)
    print("%d prototypes" % len(lines))


if __name__ == "__main__":
    main()
