"""cbev_lookahead_ex without a GPU: the entry point rejects a null handle first and every bad host argument before any
CUDA call, each with its rule; the header, the library exports and engine.EXPORTS agree; cbev_lookahead_io has the
same layout in C (g++ probe of include/cbev.h) and in the ctypes mirror."""
import ctypes as C
import os
import re
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
IO_FIELDS = ("src_info", "src_rows", "roots", "obs", "obs_bytes", "leaf_rows", "leaf_bytes", "leaf_info")


def _fake_handle():
    # a zeroed block as large as the engine struct stands in for an engine with N = 0 envs, F = 0, no ring, no
    # retreat slots, token 0 and pool epoch 0
    fake = (C.c_uint8 * (1 << 16))()
    return fake, C.addressof(fake)


def _row_bytes_of_fake():
    # header 16 + the 16 sections at A = 1, R = 0, each padded to 16 bytes; F = 0 frames
    sizes = [8 * 24, 4 * 8, 8 * 2, 8 * 12] + [8] * 7 + [4, 4, 1] + [0, 0]
    return 16 + sum((s + 15) // 16 * 16 for s in sizes)


def _ex_call(lib, handle=None, io=True, roots=True, b=4, h=8, actions=True, gamma=1.0, ret=True, steps=True,
             src=None, src_rows="ok", obs=None, obs_bytes=1 << 20, leaf=None, leaf_bytes=1 << 20, leaf_info=True):
    from carlabev_env_b200 import engine

    buf = (C.c_double * 64)()
    mem = (C.c_uint8 * 128)()
    base = (C.addressof(mem) + 15) & ~15
    ptr = {"ok": base, "none": None, "odd": base + 4, None: None}
    o = engine.CbevLookaheadOut(C.addressof(buf) if ret else None, None, C.addressof(buf) if steps else None, None,
                                None, None, None)
    li = engine.CbevSnapshotInfo()
    x = engine.CbevLookaheadIo(C.pointer(src) if src is not None else None, ptr[src_rows],
                               C.addressof(buf) if roots else None, ptr[obs], obs_bytes, ptr[leaf], leaf_bytes,
                               C.pointer(li) if leaf_info else None)
    rc = lib.cbev_lookahead_ex(handle, C.byref(x) if io else None, b, h, C.addressof(buf) if actions else None, gamma,
                               C.byref(o), None)
    return rc, lib.cbev_last_error().decode()


def _info(token=0, epoch=0, R=0, row_bytes=None, n_rows=8):
    from carlabev_env_b200 import engine

    return engine.CbevSnapshotInfo(token, epoch, R, _row_bytes_of_fake() if row_bytes is None else row_bytes, n_rows,
                                   0)


def test_null_handle_is_rejected_first():
    from carlabev_env_b200 import engine

    lib = engine.load_library()
    rc, msg = _ex_call(lib, io=False, b=0, h=0, actions=False, ret=False)
    assert rc == 1 and "null handle" in msg


def test_argument_errors_name_their_rule():
    from carlabev_env_b200 import engine

    lib = engine.load_library()
    fake, h = _fake_handle()
    cases = [
        (dict(io=False), "cbev_lookahead_ex: io is required"),
        (dict(actions=False), "cbev_lookahead_ex: actions_dev and out->ret are required"),
        (dict(ret=False), "actions_dev and out->ret are required"),
        (dict(b=0), "n_branches must be >= 1, got 0"),
        (dict(h=0), "horizon must be >= 1, got 0"),
        (dict(gamma=float("nan")), "gamma must be finite"),
        (dict(roots=False), "with NULL roots branch b starts from env b"),
        (dict(src=_info(), src_rows="none"), "src_rows is required with src_info"),
        (dict(src=_info(), src_rows="odd"), "src_rows must be 16-byte aligned"),
        (dict(src=_info(R=1)), "the src rows have 1 retreat slots, more than the engine's 0"),
        (dict(src=_info(row_bytes=16)), "src row_bytes 16 does not match"),
        (dict(src=_info(), roots=False, b=9), "branch b starts from row b, so n_branches must be <= 8 (src n_rows)"),
        (dict(src=_info(n_rows=0)), "so n_branches must be <= 0 (src n_rows)"),
        (dict(obs="odd"), "obs must be 16-byte aligned"),
        (dict(obs="ok", obs_bytes=-1), "obs holds -1 bytes"),
        (dict(leaf="ok", leaf_info=False), "leaf_info is required with leaf_rows"),
        (dict(leaf="odd"), "leaf_rows must be 16-byte aligned"),
        (dict(leaf="ok", leaf_bytes=4 * _row_bytes_of_fake() - 1), "leaf_rows holds"),
        (dict(leaf="ok", steps=False), "out->steps is required with obs or leaf_rows"),
        (dict(obs="ok", steps=False), "out->steps is required with obs or leaf_rows"),
    ]
    for kw, match in cases:
        rc, msg = _ex_call(lib, handle=h, **kw)
        assert rc == 1 and match in msg, (kw, rc, msg)
    # foreign and stale rows are state errors, refused before anything else happens
    for kw, match in [(dict(src=_info(token=7)), "the src rows were taken by another engine"),
                      (dict(src=_info(epoch=1)), "the src rows were taken under pool epoch 1, the engine is at 0")]:
        rc, msg = _ex_call(lib, handle=h, **kw)
        assert rc == 3 and match in msg, (kw, rc, msg)
    # every argument valid, frames asked for: the fake engine has no observation ring bound
    for kw in (dict(leaf="ok"), dict(obs="ok"), dict(src=_info(), leaf="ok", roots=False)):
        rc, msg = _ex_call(lib, handle=h, **kw)
        assert rc == 3 and "no observation ring bound" in msg, (kw, rc, msg)


def test_header_exports_and_engine_exports_agree():
    from carlabev_env_b200 import engine

    header = open(os.path.join(ROOT, "include", "cbev.h")).read()
    assert re.search(r"\bint cbev_lookahead_ex\(", header) and "cbev_lookahead_ex" in engine.EXPORTS
    assert "} cbev_lookahead_io;" in header
    lib_path = engine.load_library()._name
    syms = subprocess.run(["nm", "-D", "--defined-only", lib_path], capture_output=True, text=True, check=True).stdout
    assert re.search(r"\bT cbev_lookahead_ex\b", syms)


def test_lookahead_io_layout_matches_ctypes(tmp_path):
    from carlabev_env_b200 import engine

    src = tmp_path / "probe.cpp"
    body = "\n".join(f'  printf("%zu\\n", offsetof(cbev_lookahead_io, {f}));' for f in IO_FIELDS)
    src.write_text('#include <cstddef>\n#include <cstdio>\n#include "cbev.h"\nint main() {\n'
                   '  printf("%zu\\n", sizeof(cbev_lookahead_io));\n' + body + "\n  return 0;\n}\n")
    exe = tmp_path / "probe"
    subprocess.run(["g++", "-std=c++17", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    S = engine.CbevLookaheadIo
    assert got == [C.sizeof(S)] + [getattr(S, f).offset for f in IO_FIELDS]
    assert C.sizeof(S) == 64 and [f for f, _ in S._fields_] == list(IO_FIELDS)
