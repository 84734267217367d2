"""cbev_lookahead_obs and cbev_fuse_windows without a GPU: both entry points reject a null handle first and every bad
host argument before any CUDA call, each with its rule; the header, the library exports and engine.EXPORTS agree."""
import ctypes as C
import os
import re
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _fake_handle():
    # a zeroed block as large as the engine struct stands in for an engine with N = 0 envs, F = 0, no ring
    fake = (C.c_uint8 * (1 << 16))()
    return fake, C.addressof(fake)


def _obs_call(lib, handle=None, roots=True, b=4, h=8, actions=True, gamma=1.0, ret=True, steps=True, out=True,
              obs="ok", obs_bytes=1 << 20):
    from carlabev_env_b200 import engine

    buf = (C.c_double * 64)()
    win = (C.c_uint8 * 64)()
    base = (C.addressof(win) + 15) & ~15
    ptr = {"ok": base, "none": None, "odd": base + 4}[obs]
    o = engine.CbevLookaheadOut(C.addressof(buf) if ret else None, None, C.addressof(buf) if steps else None, None,
                                None, None, None)
    rc = lib.cbev_lookahead_obs(handle, C.addressof(buf) if roots else None, b, h,
                                C.addressof(buf) if actions else None, gamma, C.byref(o) if out else None, ptr,
                                obs_bytes, None)
    return rc, lib.cbev_last_error().decode()


def _fuse_call(lib, handle=None, mode=1, windows="ok", n=4, out="ok"):
    win = (C.c_uint8 * 64)()
    base = (C.addressof(win) + 15) & ~15
    ptrs = {"ok": base, "none": None, "odd": base + 8}
    rc = lib.cbev_fuse_windows(handle, mode, ptrs[windows], n, ptrs[out], None)
    return rc, lib.cbev_last_error().decode()


def test_null_handle_is_rejected_first():
    from carlabev_env_b200 import engine

    lib = engine.load_library()
    rc, msg = _obs_call(lib, b=0, h=0, actions=False, ret=False, steps=False, obs="none", obs_bytes=-1)
    assert rc == 1 and "null handle" in msg
    rc, msg = _fuse_call(lib, mode=0, windows="none", n=0, out="none")
    assert rc == 1 and "null handle" in msg


def test_lookahead_obs_argument_errors_name_their_rule():
    from carlabev_env_b200 import engine

    lib = engine.load_library()
    fake, h = _fake_handle()
    cases = [
        (dict(actions=False), "cbev_lookahead_obs: actions_dev and out->ret are required"),
        (dict(ret=False), "actions_dev and out->ret are required"),
        (dict(out=False), "actions_dev and out->ret are required"),
        (dict(b=0), "n_branches must be >= 1, got 0"),
        (dict(h=0), "horizon must be >= 1, got 0"),
        (dict(gamma=float("nan")), "gamma must be finite"),
        (dict(roots=False), "with NULL roots branch b starts from env b"),
        (dict(steps=False), "out->steps is required"),
        (dict(obs="none"), "obs_dev is required"),
        (dict(obs="odd"), "obs_dev must be 16-byte aligned"),
        (dict(obs_bytes=-1), "obs_dev holds -1 bytes"),
    ]
    for kw, match in cases:
        rc, msg = _obs_call(lib, handle=h, **kw)
        assert rc == 1 and match in msg, (kw, rc, msg)
    # every argument valid: the fake engine has no observation ring bound
    rc, msg = _obs_call(lib, handle=h)
    assert rc == 3 and "no observation ring bound" in msg, (rc, msg)


def test_fuse_windows_argument_errors_name_their_rule():
    from carlabev_env_b200 import engine

    lib = engine.load_library()
    fake, h = _fake_handle()
    cases = [
        (dict(windows="none"), "null windows or output"),
        (dict(out="none"), "null windows or output"),
        (dict(windows="odd"), "16-byte aligned"),
        (dict(out="odd"), "16-byte aligned"),
        (dict(n=0), "n must be >= 1, got 0"),
        (dict(mode=0), "bad fusion mode 0"),
        (dict(mode=3), "bad fusion mode 3"),
        (dict(), "requires frame_stack >= 3"),  # the zeroed config: semantic masks, frame_stack 0
    ]
    for kw, match in cases:
        rc, msg = _fuse_call(lib, handle=h, **kw)
        assert rc == 1 and match in msg, (kw, rc, msg)


def test_header_exports_and_engine_exports_agree():
    from carlabev_env_b200 import engine

    header = open(os.path.join(ROOT, "include", "cbev.h")).read()
    lib_path = engine.load_library()._name
    syms = subprocess.run(["nm", "-D", "--defined-only", lib_path], capture_output=True, text=True, check=True).stdout
    for name in ("cbev_lookahead_obs", "cbev_fuse_windows"):
        assert re.search(rf"\bint {name}\(", header), name
        assert name in engine.EXPORTS, name
        assert re.search(rf"\bT {name}\b", syms), name
