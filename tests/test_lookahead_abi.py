"""cbev_lookahead without a GPU: the entry point rejects a null handle and bad host arguments before any CUDA call,
each with its rule; the header, the library exports and engine.EXPORTS agree; cbev_lookahead_out has the same layout
in C (g++ probe of include/cbev.h) and in the ctypes mirror."""
import ctypes as C
import os
import re
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIELDS = ("ret", "reward", "steps", "terminated", "truncated", "cause", "hero")


def _call(lib, handle=None, roots=None, b=4, h=8, actions=True, gamma=1.0, ret=True, out=True):
    from carlabev_env_b200 import engine

    buf = (C.c_double * 64)()
    o = engine.CbevLookaheadOut(C.addressof(buf) if ret else None, None, None, None, None, None, None)
    rc = lib.cbev_lookahead(handle, roots, b, h, C.addressof(buf) if actions else None, gamma,
                            C.byref(o) if out else None, None)
    return rc, lib.cbev_last_error().decode()


def test_null_handle_is_rejected_first():
    from carlabev_env_b200 import engine

    lib = engine.load_library()
    rc, msg = _call(lib, b=0, h=0, actions=False, ret=False)
    assert rc == 1 and "null handle" in msg


def test_argument_errors_name_their_rule():
    """A dummy non-null handle: every one of these checks runs before the handle is dereferenced for CUDA work."""
    from carlabev_env_b200 import engine

    lib = engine.load_library()
    # a zeroed block as large as the engine struct stands in for an engine with N = 0 envs
    fake = (C.c_uint8 * (1 << 16))()
    h = C.addressof(fake)
    cases = [
        (dict(actions=False), "actions_dev and out->ret are required"),
        (dict(ret=False), "actions_dev and out->ret are required"),
        (dict(out=False), "actions_dev and out->ret are required"),
        (dict(b=0), "n_branches must be >= 1, got 0"),
        (dict(h=0), "horizon must be >= 1, got 0"),
        (dict(gamma=float("nan")), "gamma must be finite"),
        (dict(gamma=float("inf")), "gamma must be finite"),
        (dict(b=4), "with NULL roots branch b starts from env b"),
    ]
    for kw, match in cases:
        rc, msg = _call(lib, handle=h, **kw)
        assert rc == 1 and match in msg, (kw, rc, msg)


def test_header_exports_and_engine_exports_agree():
    from carlabev_env_b200 import engine

    header = open(os.path.join(ROOT, "include", "cbev.h")).read()
    assert re.search(r"\bcbev_lookahead\(", header) and "cbev_lookahead" in engine.EXPORTS
    assert not re.search(r"cbev_lookahead_out\s*\(", header)
    assert "} cbev_lookahead_out;" in header
    lib_path = engine.load_library()._name
    syms = subprocess.run(["nm", "-D", "--defined-only", lib_path], capture_output=True, text=True, check=True).stdout
    assert re.search(r"\bT cbev_lookahead\b", syms)


def test_lookahead_out_layout_matches_ctypes(tmp_path):
    from carlabev_env_b200 import engine

    src = tmp_path / "probe.cpp"
    body = "\n".join(f'  printf("%zu\\n", offsetof(cbev_lookahead_out, {f}));' for f in FIELDS)
    src.write_text('#include <cstddef>\n#include <cstdio>\n#include "cbev.h"\nint main() {\n'
                   '  printf("%zu\\n", sizeof(cbev_lookahead_out));\n' + body + "\n  return 0;\n}\n")
    exe = tmp_path / "probe"
    subprocess.run(["g++", "-std=c++17", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    S = engine.CbevLookaheadOut
    assert got == [C.sizeof(S)] + [getattr(S, f).offset for f in FIELDS]
    assert C.sizeof(S) == 56 and [f for f, _ in S._fields_] == list(FIELDS)
