"""Record the facts tests/test_shim_interfaces.py needs from the reference's Fortran sources.

    python tests/golden/make_reference_src.py <reference checkout>/src

Writes reference_src.json next to this file:
  system_t, int_store_t  component names of the two derived types (src/system.f90, src/integrals.f90);
  modules                for every module shim/afesp_gpu.f90 imports with `use <module>, only:`, the imported names the
                         module's source defines;
  strings                for src/ccsd.f90 and src/mp2.f90, the string literals of the shim that occur in that file.
The reference's sources are not part of this project, so the test reads only that file.
"""
import json
import os
import re
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SHIM = os.path.join(HERE, "..", "..", "shim", "afesp_gpu.f90")
MODULE_FILES = {"const": "const.F90"}


def _code(text):
    """Source lines with comments removed (a `!` inside a string literal is kept)."""
    out = []
    for line in text.splitlines():
        quote = None
        for k, ch in enumerate(line):
            if quote:
                quote = None if ch == quote else quote
            elif ch in "'\"":
                quote = ch
            elif ch == "!":
                line = line[:k]
                break
        out.append(line)
    return out


def type_components(text, name):
    """Component names declared (`<type-spec> [, attrs] :: a, b(:), c = 0`) between `type <name>` and `end type`."""
    body = re.split(r"^\s*type\s*(?:,[^:]*)?(?:::)?\s*%s\b" % name, "\n".join(_code(text)), flags=re.I | re.M)[1]
    body = re.split(r"^\s*end\s*type", body, flags=re.I | re.M)[0]
    names = set()
    for line in body.replace("&\n", " ").splitlines():
        if "::" not in line:
            continue
        depth, item = 0, ""
        for ch in line.split("::", 1)[1] + ",":
            depth += (ch in "([") - (ch in ")]")
            if ch == "," and depth == 0:
                m = re.match(r"\s*(\w+)", item)
                if m:
                    names.add(m.group(1).lower())
                item = ""
            else:
                item += ch
    return sorted(names)


def main(src):
    shim = open(SHIM).read()
    read = lambda f: open(os.path.join(src, f)).read()
    facts = {"source": "extracted from the reference's src/ by tests/golden/make_reference_src.py",
             "system_t": type_components(read("system.f90"), "system_t"),
             "int_store_t": type_components(read("integrals.f90"), "int_store_t"), "modules": {}, "strings": {}}
    for mod, names in re.findall(r"use (\w+), only: ([\w, =>]+)", shim):
        if mod in ("iso_c_binding", "iso_fortran_env"):
            continue
        text = read(MODULE_FILES.get(mod, mod + ".f90")).lower()
        found = {nm.split("=>")[-1].strip().lower() for nm in names.split(",")}
        known = set(facts["modules"].get(mod, [])) | {nm for nm in found if re.search(r"\b%s\b" % nm, text)}
        facts["modules"][mod] = sorted(known)
    literals = set(re.findall(r"'([^'\n]+)'", shim)) | set(re.findall(r'"([^"\n]+)"', shim))
    for f in ("ccsd.f90", "mp2.f90"):
        text = read(f)
        facts["strings"][f] = sorted(s for s in literals if s.strip() and s in text)
    with open(os.path.join(HERE, "reference_src.json"), "w") as fh:
        json.dump(facts, fh, indent=1)
        fh.write("\n")


if __name__ == "__main__":
    main(sys.argv[1])
