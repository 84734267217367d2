"""Same-step auto-reset without a GPU: the header defines CBEV_AUTORESET_SAME_STEP and declares cbev_bind_final_obs,
the header, the library exports and engine.EXPORTS agree, the bind call rejects a null handle, the ABI sizes and version
are unchanged, and make_env rejects the two unsupported combinations before any engine exists."""
import ctypes as C
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.abspath(os.path.dirname(__file__)))


def test_header_defines_the_mode_and_declares_the_bind_call():
    from carlabev_env_b200 import engine

    header = open(os.path.join(ROOT, "include", "cbev.h")).read()
    assert re.search(r"#define CBEV_AUTORESET_SAME_STEP 2\b", header)
    assert re.search(r"int cbev_bind_final_obs\(cbev_handle h, void\* final_dev, int64_t bytes\);", header)
    assert engine.AUTORESET_SAME_STEP == 2


def test_header_exports_and_engine_exports_agree():
    from carlabev_env_b200 import engine

    header = open(os.path.join(ROOT, "include", "cbev.h")).read()
    declared = set(re.findall(r"\b(?:int|int64_t|const char\*)\s+(cbev_\w+)\(", header))
    syms = subprocess.run(["nm", "-D", "--defined-only", engine.load_library()._name], capture_output=True, text=True,
                          check=True).stdout
    exported = set(re.findall(r"\bT (cbev_\w+)\b", syms))
    assert "cbev_bind_final_obs" in declared and "cbev_bind_final_obs" in engine.EXPORTS
    assert declared == exported == set(engine.EXPORTS), (declared ^ exported, exported ^ set(engine.EXPORTS))


def test_bind_rejects_a_null_handle():
    from carlabev_env_b200 import engine

    lib = engine.load_library()
    buf = (C.c_uint8 * 64)()
    assert lib.cbev_bind_final_obs(None, C.addressof(buf), 64) == 1
    assert "null handle" in lib.cbev_last_error().decode()


def test_abi_sizes_and_version_are_unchanged():
    from carlabev_env_b200 import engine

    lib = engine.load_library()
    sizes = [C.c_int32(), C.c_int32(), C.c_int32()]
    assert lib.cbev_abi_sizes(*[C.byref(v) for v in sizes]) == 0
    got = tuple(v.value for v in sizes)
    assert got == (C.sizeof(engine.CbevConfig), C.sizeof(engine.CbevPoolDesc), C.sizeof(engine.CbevStepOut))
    assert got[2] == 48 and lib.cbev_version() == 201


def test_make_env_rejects_video_and_device_side_fusion():
    from carlabev_env_b200.config import EnvConfig, RunConfig
    from carlabev_env_b200.vector_env import make_env

    with pytest.raises(ValueError, match="capture_video"):
        make_env(RunConfig(env=EnvConfig(), num_envs=2, capture_video=True), autoreset="same_step")
    fused = RunConfig(env=EnvConfig(temporal_fusion_mode="vehicle_temporal"), num_envs=2)
    with pytest.raises(ValueError, match="host_infos=True"):
        make_env(fused, autoreset="same_step", host_infos=False)
