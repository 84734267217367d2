"""The reward parameters of cbev_config without a GPU: every CaRL and shaping field sits at the same offset in C (g++
probe of include/cbev.h) and in the ctypes mirror `CbevConfig`, and every key of CARL_DEFAULTS / SHAPING_DEFAULTS --
the names `Engine(reward_params=...)` accepts -- is a field of the matching C type.  Two same-typed fields swapped in
the mirror keep `sizeof` equal; they move an offset here."""
import ctypes as C
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _fields():
    from carlabev_env_b200 import engine as E

    return [f for f, _ in E.CbevConfig._fields_]


def test_cbev_config_layout_matches_ctypes(tmp_path):
    from carlabev_env_b200 import engine as E

    fields = _fields()
    src = tmp_path / "probe.cpp"
    body = "\n".join(f'  printf("%zu %zu\\n", offsetof(cbev_config, {f}), sizeof(((cbev_config*)0)->{f}));'
                     for f in fields)
    src.write_text('#include <cstddef>\n#include <cstdio>\n#include "cbev.h"\nint main() {\n'
                   '  printf("%zu 0\\n", sizeof(cbev_config));\n' + body + "\n  return 0;\n}\n")
    exe = tmp_path / "probe"
    subprocess.run(["g++", "-std=c++17", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split("\n")
    got = [tuple(int(v) for v in line.split()) for line in out if line.strip()]
    S = E.CbevConfig
    assert got[0][0] == C.sizeof(S)
    want = [(getattr(S, f).offset, getattr(S, f).size) for f in fields]
    bad = [(f, g, w) for f, g, w in zip(fields, got[1:], want) if g != w]
    assert not bad, f"(field, C offset/size, ctypes offset/size): {bad}"


def _header_fields():
    """(name, C type) of every cbev_config member, in the header's order."""
    import re

    header = open(os.path.join(ROOT, "include", "cbev.h")).read()
    body = header[header.index("typedef struct {", header.index("---- configuration")):header.index("} cbev_config;")]
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S).split("{", 1)[1]
    out = []
    for decl in body.split(";"):
        if decl.strip():
            ctype, rest = decl.split(None, 1)
            out += [(re.sub(r"\[.*\]", "", n).strip(), ctype) for n in rest.split(",")]
    return out


def test_cbev_config_names_and_types_match_the_header():
    """The probe above proves offsets for the fields the mirror names; this proves it names all of them, in order,
    each with the ctypes type of its C declaration."""
    from carlabev_env_b200 import engine as E

    ctypes_of = {"int32_t": C.c_int32, "double": C.c_double, "uint64_t": C.c_uint64, "float": C.c_float}
    hdr = _header_fields()
    assert [n for n, _ in hdr] == _fields()
    for (name, ctype), (_, t) in zip(hdr, E.CbevConfig._fields_):
        assert (t._type_ if issubclass(t, C.Array) else t) is ctypes_of[ctype], (name, ctype, t)


def test_reward_defaults_are_cbev_config_fields_of_the_matching_type():
    from carlabev_env_b200.config import CARL_DEFAULTS, SHAPING_DEFAULTS

    types = dict(_header_fields())
    assert not set(CARL_DEFAULTS) & set(SHAPING_DEFAULTS)
    for k, v in {**CARL_DEFAULTS, **SHAPING_DEFAULTS}.items():
        assert k in types, k
        want = "int32_t" if isinstance(v, int) and not isinstance(v, bool) else "double"
        assert types[k] == want, (k, v, types[k])
    # the C block of each family holds exactly its defaults' keys
    fields = _fields()
    carl = fields[fields.index("lane_center_exponent"):fields.index("ttc_penalty_floor") + 1]
    shaping = fields[fields.index("max_actions"):fields.index("lat_small") + 1]
    assert sorted(carl) == sorted(CARL_DEFAULTS)
    assert sorted(shaping) == sorted(SHAPING_DEFAULTS)
