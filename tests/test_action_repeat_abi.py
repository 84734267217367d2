"""cbev_set_action_repeat without a GPU: a null handle and out-of-range repeats are rejected, each with its rule; the
header, the library exports and engine.EXPORTS agree; the ABI struct sizes are unchanged."""
import ctypes as C
import os
import re
import subprocess

ROOT = os.path.dirname(os.path.abspath(os.path.dirname(__file__)))


def test_null_handle_is_rejected():
    from carlabev_env_b200 import engine

    lib = engine.load_library()
    assert lib.cbev_set_action_repeat(None, 4) == 1
    assert "null handle" in lib.cbev_last_error().decode()


def test_repeat_outside_1_to_64_is_rejected_with_its_rule():
    from carlabev_env_b200 import engine

    lib = engine.load_library()
    fake = (C.c_uint8 * (1 << 16))()  # the range check runs before the engine is used
    for k in (0, -1, 65):
        assert lib.cbev_set_action_repeat(C.addressof(fake), k) == 1, k
        assert f"repeat must lie in [1, 64], got {k}" in lib.cbev_last_error().decode()
    assert engine.MAX_ACTION_REPEAT == 64


def test_header_exports_and_engine_exports_agree():
    from carlabev_env_b200 import engine

    header = open(os.path.join(ROOT, "include", "cbev.h")).read()
    assert re.search(r"int cbev_set_action_repeat\(cbev_handle h, int32_t repeat\);", header)
    assert re.search(r"#define CBEV_MAX_ACTION_REPEAT 64\b", header)
    assert "cbev_set_action_repeat" in engine.EXPORTS
    syms = subprocess.run(["nm", "-D", "--defined-only", engine.load_library()._name], capture_output=True, text=True,
                          check=True).stdout
    assert re.search(r"\bT cbev_set_action_repeat\b", syms)


def test_abi_sizes_are_unchanged():
    from carlabev_env_b200 import engine

    lib = engine.load_library()
    sizes = [C.c_int32(), C.c_int32(), C.c_int32()]
    assert lib.cbev_abi_sizes(*[C.byref(v) for v in sizes]) == 0
    got = tuple(v.value for v in sizes)
    assert got == (C.sizeof(engine.CbevConfig), C.sizeof(engine.CbevPoolDesc), C.sizeof(engine.CbevStepOut))
    assert got[2] == 48 and lib.cbev_version() == 201
