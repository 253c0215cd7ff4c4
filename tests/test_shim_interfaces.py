"""Static cross-check of the Fortran side of the boundary (no Fortran compiler exists in this image, SURVEY.md K5).

shim/afesp_gpu.f90 is delivered as source only, so what CAN be verified without compiling it is verified here:
  * every ISO_C_BINDING interface in the shim names a function include/afesp_gpu.h declares, with the same number of
    arguments, each passed the way the C prototype expects (by value / by reference) and with the matching C type;
  * the shim covers every export of the header;
  * free-form source limits (132 columns, continuation markers) hold;
  * every component of the reference's derived types the wrappers touch (sys%..., int_store%...), every module entity
    they import and every printed line they keep exists in the reference's sources, as recorded in
    tests/golden/reference_src.json (tests/golden/make_reference_src.py); the printed lines also appear in the outputs
    the reference shipped (tests/golden/*_out.txt).
"""
import json
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SHIM = os.path.join(ROOT, "shim", "afesp_gpu.f90")
HEADER = os.path.join(ROOT, "include", "afesp_gpu.h")
GOLDEN = os.path.join(ROOT, "tests", "golden")


# ------------------------------------------------------------------------------------------------ C prototypes
def _c_prototypes():
    text = open(HEADER).read()
    text = re.sub(r"/\*.*?\*/", " ", text, flags=re.S)
    protos = {}
    for ret, name, args in re.findall(r"\b(const\s+char\s*\*|int)\s+(afesp_gpu_\w+)\s*\(([^)]*)\)\s*;", text):
        params = []
        for a in [x.strip() for x in args.split(",") if x.strip()]:
            a = re.sub(r"\s+", " ", a)
            is_array = "[" in a
            a_type = re.sub(r"\[[^\]]*\]", "", a)
            a_type = re.sub(r"\b\w+$", "", a_type).strip() if not a_type.endswith("*") else a_type   # drop the name
            stars = a_type.count("*") + (1 if is_array else 0)
            base = a_type.replace("*", "").replace("const", "").strip()
            if base == "afesp_handle":
                base, stars = "void", stars + 1
            params.append((base, stars))
        protos[name] = ("ptr" if "char" in ret else "int", params)
    return protos


# ------------------------------------------------------------------------------------------------ Fortran interfaces
def _joined_lines(text):
    """Free-form source with `&` continuations joined and comments stripped."""
    out, cur = [], ""
    for raw in text.splitlines():
        line = raw.split("!")[0].rstrip() if "'" not in raw.split("!")[0] or raw.count("'") % 2 == 0 else raw.rstrip()
        if not line.strip():
            continue
        if cur:
            line = line.lstrip()
            if line.startswith("&"):
                line = line[1:]
        if line.endswith("&"):
            cur += line[:-1] + " "
            continue
        out.append(cur + line)
        cur = ""
    assert not cur, "dangling continuation"
    return out


_F_TYPES = {"integer(c_int)": "int", "integer(c_long_long)": "long long", "real(c_double)": "double",
            "character(kind=c_char)": "char", "type(c_ptr)": "c_ptr"}


def _shim_interfaces():
    lines = _joined_lines(open(SHIM).read())
    start = next(i for i, l in enumerate(lines) if l.strip() == "interface")
    end = next(i for i, l in enumerate(lines) if l.strip() == "end interface")
    out, cur = {}, None
    for l in lines[start + 1:end]:
        s = l.strip()
        m = re.match(r"(integer\(c_int\)|type\(c_ptr\))\s+function\s+(\w+)\s*\(([^)]*)\)\s*bind\(C,\s*name='(\w+)'\)", s)
        if m:
            cur = {"ret": "int" if m.group(1).startswith("integer") else "ptr",
                   "args": [a.strip() for a in m.group(3).split(",") if a.strip()], "bind": m.group(4), "decl": {},
                   "imports": set()}
            out[m.group(2)] = cur
            continue
        if s == "end function":
            cur = None
            continue
        assert cur is not None, f"statement outside a function interface: {s}"
        if s.startswith("import ::"):
            cur["imports"] |= {x.strip() for x in s[len("import ::"):].split(",")}
            continue
        m = re.match(r"(\w+\([\w=]+\))\s*((?:,\s*[\w]+(?:\([^)]*\))?\s*)*)::\s*(.*)$", s)
        assert m, f"unparsed declaration: {s}"
        ftype, attrs, names = m.group(1), m.group(2), m.group(3)
        assert ftype in _F_TYPES, ftype
        attrs = [a.strip() for a in attrs.split(",") if a.strip()]
        for nm in [x.strip() for x in names.split(",")]:
            cur["decl"][nm.lower()] = (ftype, attrs)
    return out


def test_every_shim_interface_matches_its_c_prototype():
    protos = _c_prototypes()
    ifaces = _shim_interfaces()
    assert len(protos) >= 35 and "afesp_gpu_ccsd_iterate" in protos
    for fname, it in ifaces.items():
        assert it["bind"] == fname, (fname, it["bind"])
        assert fname in protos, f"{fname}: not declared in include/afesp_gpu.h"
        ret, params = protos[fname]
        assert it["ret"] == ret, (fname, "return type")
        assert len(it["args"]) == len(params), (fname, it["args"], params)
        used_kinds = set()
        for arg, (cbase, stars) in zip(it["args"], params):
            assert arg.lower() in it["decl"], (fname, arg, "dummy argument has no declaration")
            ftype, attrs = it["decl"][arg.lower()]
            used_kinds.add(re.search(r"c_\w+", ftype).group(0))
            by_value = "value" in attrs
            if _F_TYPES[ftype] == "c_ptr":
                # type(c_ptr), value = any data pointer;  type(c_ptr), intent(out) = pointer to pointer (afesp_handle*)
                assert stars == (1 if by_value else 2), (fname, arg, cbase, stars)
                continue
            assert _F_TYPES[ftype] == cbase, (fname, arg, ftype, cbase)
            if by_value:
                assert stars == 0, (fname, arg, "passed by value but the C side expects a pointer")
                assert not any(a.startswith("dimension") or a.startswith("intent(out") for a in attrs), (fname, arg)
            else:
                assert stars == 1, (fname, arg, "passed by reference but the C side expects a value")
        # `import ::` must bring in exactly the kinds the declarations use (+ the return type's)
        used_kinds.add("c_int" if it["ret"] == "int" else "c_ptr")
        assert used_kinds <= it["imports"], (fname, used_kinds - it["imports"])
        # dummy arguments are case-insensitive in Fortran: no two may collide
        assert len({a.lower() for a in it["args"]}) == len(it["args"]), (fname, "argument names collide ignoring case")


def test_shim_covers_every_export_of_the_header():
    assert set(_shim_interfaces()) == set(_c_prototypes())


def test_shim_respects_free_form_source_limits():
    depth = 0
    for k, raw in enumerate(open(SHIM).read().splitlines(), 1):
        assert len(raw) <= 132, f"line {k} has {len(raw)} columns (free-form limit 132)"
        assert "\t" not in raw, f"line {k}: tab character"
        s = raw.split("!")[0].strip().lower()
        if re.match(r"(subroutine|module)\s+\w+", s) and not s.startswith("module procedure"):
            depth += 1
        if re.match(r"end\s+(subroutine|module)\b", s):
            depth -= 1
    assert depth == 0, "unbalanced subroutine/module blocks"


def test_wrappers_check_every_status():
    """Each call into the library is wrapped in check(...) (status -> error(), src/error_handling.f90:7-20) or its status is
    kept in a variable that is checked."""
    body = open(SHIM).read().split("contains", 1)[1]
    joined = "\n".join(_joined_lines(body))
    calls = re.findall(r"(\w[\w ]*=\s*)?(?:call check\(\s*)?(afesp_gpu_\w+)\(", joined)
    assert len(calls) >= 12
    for line in joined.splitlines():
        for m in re.finditer(r"afesp_gpu_(?!last_error)\w+\(", line):
            pre = line[:m.start()]
            assert "check(" in pre or re.search(r"\brc\s*=\s*$", pre), f"status of this call is dropped: {line.strip()}"
    assert re.search(r"call check\(rc,", joined), "the kept status rc is never checked"


def test_wrappers_only_touch_entities_the_reference_defines():
    shim = open(SHIM).read()
    ref = json.load(open(os.path.join(GOLDEN, "reference_src.json")))
    for comp in sorted(set(re.findall(r"\bsys%(\w+)", shim))):
        assert comp.lower() in ref["system_t"], f"system_t has no component {comp}"
    for comp in sorted(set(re.findall(r"\bint_store%(\w+)", shim))):
        assert comp.lower() in ref["int_store_t"], f"int_store_t has no component {comp}"
    # module entities imported with `use <module>, only:`
    for mod, names in re.findall(r"use (\w+), only: ([\w, =>]+)", shim):
        if mod in ("iso_c_binding", "iso_fortran_env"):
            continue
        for nm in [x.split("=>")[-1].strip() for x in names.split(",")]:
            assert nm.lower() in ref["modules"].get(mod, []), f"module {mod} has no entity {nm}"
    # the printed lines the wrappers keep are the reference's own format strings
    printed = {"mp2.f90": ["Performing AO to MO ERI transformation...", "Calculating MP2 energy...",
                           "MP2 correlation energy (Hartree):"],
               "ccsd.f90": ["Convergence reached within tolerance.", "Final CCSD Energy (Hartree):", "T1 diagnostic:",
                            "Forming antisymmetrised spinorbital ERIs...",
                            "Checking that the permuational symmetry of the antisymmetrised integrals hold...",
                            "Unrestricted CCSD(T) correlation energy (Hartree):"]}
    kept = {"ccsd.f90": ["Permutational symmetry of antisymmetrised integrals does not hold",   # error path
                         "(1X, I9, 3X, F15.12, 3X, F15.12, 3X, F15.12, 3X, F8.6)"]}         # iteration-table format
    shipped = "".join(open(os.path.join(GOLDEN, f)).read() for f in sorted(os.listdir(GOLDEN)) if f.endswith("_out.txt"))
    for fname in ("mp2.f90", "ccsd.f90"):
        for text in printed[fname] + kept.get(fname, []):
            assert text in shim and text in ref["strings"][fname], (fname, text)
        for text in printed[fname]:
            assert text in shipped, text
