"""Parser of include/sylow_b200.h: its status and hash constants and the prototype of every exported function.
The ctypes binding (_lib.py) and the Rust bindings generator (tools/gen_rust_ffi.py) both read the C ABI from here,
so the header is the only place it is written down."""
from __future__ import annotations

import os
import re
from typing import List, NamedTuple, Tuple

HEADER = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "sylow_b200.h")


class CType(NamedTuple):
    """`const uint8_t*` is CType("uint8_t", True, 1): the base type, whether the innermost pointee is const, and the
    pointer depth."""
    base: str
    const: bool
    stars: int


def ctype(decl: str) -> CType:
    words = decl.replace("*", " ").split()
    base = [w for w in words if w != "const"]
    assert len(base) == 1, decl
    return CType(base[0], "const" in words, decl.count("*"))


def parse(header: str = HEADER) -> Tuple[List[Tuple[str, str]], List[Tuple[str, List[Tuple[str, CType]], CType]]]:
    """([(constant, value)], [(function, [(parameter, type)], return type)]), both in header order.  An array
    parameter (`uint8_t out[384]`) is the pointer it decays to."""
    text = re.sub(r"/\*.*?\*/", " ", open(header).read(), flags=re.S)
    text = re.sub(r"//[^\n]*", " ", text)
    consts = re.findall(r"\b(SYLOW_B200_[A-Z0-9_]+)\s*=\s*(-?\d+)", text)  # the status enum
    consts += re.findall(r"#define\s+(SYLOW_B200_[A-Z0-9_]+)\s+(-?\d+)", text)
    funcs = []
    for ret, name, args in re.findall(r"([A-Za-z_][A-Za-z0-9_ ]*?\**)\s*\b(sylow_b200_[a-z0-9_]+)\s*\(([^;{]*?)\)\s*;", text):
        params = []
        for a in [x.strip() for x in args.replace("\n", " ").split(",") if x.strip()]:
            if a == "void":
                continue
            m = re.match(r"(.*?)([A-Za-z_][A-Za-z0-9_]*)\s*(\[\s*\d*\s*\])?$", a)
            decl, pname, arr = m.group(1), m.group(2), m.group(3)
            params.append((pname, ctype(decl + "*" if arr else decl)))
        funcs.append((name, params, ctype(ret)))
    return consts, funcs
