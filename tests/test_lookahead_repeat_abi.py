"""cbev_lookahead_repeat without a GPU: the entry point rejects a null handle first, a repeat outside [1, 64] and every
bad host argument of cbev_lookahead_ex before any CUDA call, each with its rule naming the new entry point; the
header, the library exports and engine.EXPORTS agree; the ABI sizes are unchanged; Engine.lookahead(repeat=) raises
the ValueError of set_action_repeat."""
import ctypes as C
import os
import re
import subprocess

import pytest

from test_lookahead_rows_abi import _fake_handle, _info, _row_bytes_of_fake

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _rep_call(lib, handle=None, repeat=4, io=True, roots=True, b=4, h=8, actions=True, gamma=1.0, ret=True,
              steps=True, src=None, src_rows="ok", obs=None, obs_bytes=1 << 20, leaf=None, leaf_bytes=1 << 20,
              leaf_info=True):
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
    rc = lib.cbev_lookahead_repeat(handle, C.byref(x) if io else None, b, h, repeat,
                                   C.addressof(buf) if actions else None, gamma, C.byref(o), None)
    return rc, lib.cbev_last_error().decode()


def test_null_handle_is_rejected_first():
    from carlabev_env_b200 import engine

    lib = engine.load_library()
    rc, msg = _rep_call(lib, repeat=0, io=False, b=0, h=0, actions=False, ret=False)
    assert rc == 1 and "null handle" in msg


def test_repeat_outside_1_to_64_is_rejected_with_its_rule():
    from carlabev_env_b200 import engine

    lib = engine.load_library()
    fake, h = _fake_handle()
    for k in (0, -1, 65):
        rc, msg = _rep_call(lib, handle=h, repeat=k)
        assert rc == 1 and f"cbev_lookahead_repeat: repeat must lie in [1, 64], got {k}" in msg, (k, rc, msg)
    # 1 and 64 pass the range check and stop at the next rule (the fake engine has no ring for the frames)
    for k in (1, 64):
        rc, msg = _rep_call(lib, handle=h, repeat=k, obs="ok")
        assert rc == 3 and "cbev_lookahead_repeat: no observation ring bound" in msg, (k, rc, msg)


def test_inherited_argument_errors_name_their_rule():
    from carlabev_env_b200 import engine

    lib = engine.load_library()
    fake, h = _fake_handle()
    cases = [
        (dict(io=False), "cbev_lookahead_repeat: io is required"),
        (dict(actions=False), "cbev_lookahead_repeat: actions_dev and out->ret are required"),
        (dict(ret=False), "actions_dev and out->ret are required"),
        (dict(b=0), "n_branches must be >= 1, got 0"),
        (dict(h=0), "horizon must be >= 1, got 0"),
        (dict(gamma=float("inf")), "gamma must be finite"),
        (dict(roots=False), "with NULL roots branch b starts from env b"),
        (dict(src=_info(), src_rows="none"), "src_rows is required with src_info"),
        (dict(src=_info(), src_rows="odd"), "src_rows must be 16-byte aligned"),
        (dict(src=_info(R=1)), "the src rows have 1 retreat slots, more than the engine's 0"),
        (dict(src=_info(row_bytes=16)), "src row_bytes 16 does not match"),
        (dict(src=_info(), roots=False, b=9), "branch b starts from row b, so n_branches must be <= 8 (src n_rows)"),
        (dict(obs="odd"), "obs must be 16-byte aligned"),
        (dict(obs="ok", obs_bytes=-1), "obs holds -1 bytes"),
        (dict(leaf="ok", leaf_info=False), "leaf_info is required with leaf_rows"),
        (dict(leaf="odd"), "leaf_rows must be 16-byte aligned"),
        (dict(leaf="ok", leaf_bytes=4 * _row_bytes_of_fake() - 1), "leaf_rows holds"),
        (dict(leaf="ok", steps=False), "out->steps is required with obs or leaf_rows"),
    ]
    for kw, match in cases:
        rc, msg = _rep_call(lib, handle=h, **kw)
        assert rc == 1 and match in msg and msg.startswith("cbev_lookahead_repeat"), (kw, rc, msg)
    for kw, match in [(dict(src=_info(token=7)), "the src rows were taken by another engine"),
                      (dict(src=_info(epoch=1)), "the src rows were taken under pool epoch 1, the engine is at 0"),
                      (dict(leaf="ok"), "no observation ring bound")]:
        rc, msg = _rep_call(lib, handle=h, **kw)
        assert rc == 3 and match in msg, (kw, rc, msg)


def test_header_exports_and_engine_exports_agree():
    from carlabev_env_b200 import engine

    header = open(os.path.join(ROOT, "include", "cbev.h")).read()
    assert re.search(r"int cbev_lookahead_repeat\(cbev_handle h, const cbev_lookahead_io\* io, int32_t n_branches, "
                     r"int32_t horizon,\s+int32_t repeat, const void\* actions_dev, double gamma, "
                     r"const cbev_lookahead_out\* out,\s+void\* stream\);", header)
    assert "cbev_lookahead_repeat" in engine.EXPORTS
    syms = subprocess.run(["nm", "-D", "--defined-only", engine.load_library()._name], capture_output=True, text=True,
                          check=True).stdout
    assert re.search(r"\bT cbev_lookahead_repeat\b", syms)
    declared = set(re.findall(r"\bint(?:64_t)?\s+(cbev_\w+)\(", header))
    assert set(engine.EXPORTS) <= declared | {"cbev_last_error", "cbev_version", "cbev_abi_sizes"}


def test_abi_sizes_are_unchanged():
    from carlabev_env_b200 import engine

    lib = engine.load_library()
    sizes = [C.c_int32(), C.c_int32(), C.c_int32()]
    assert lib.cbev_abi_sizes(*[C.byref(v) for v in sizes]) == 0
    got = tuple(v.value for v in sizes)
    assert got == (C.sizeof(engine.CbevConfig), C.sizeof(engine.CbevPoolDesc), C.sizeof(engine.CbevStepOut))
    assert got[2] == 48 and lib.cbev_version() == 201
    assert C.sizeof(engine.CbevLookaheadIo) == 64 and C.sizeof(engine.CbevLookaheadOut) == 56


@pytest.mark.parametrize("bad", [0, 65, -3, 2.5, True, False])
def test_python_repeat_errors_match_set_action_repeat(bad):
    """The range and type checks run before the engine is used, so no engine (and no GPU) is needed."""
    from carlabev_env_b200 import engine

    with pytest.raises(ValueError) as ref:
        engine.Engine.set_action_repeat(None, bad)
    with pytest.raises(ValueError) as got:
        engine.Engine.lookahead(None, None, repeat=bad)
    assert str(got.value) == str(ref.value) == f"action repeat must be an integer in [1, 64], got {bad!r}"
