"""Snapshot / restore (cbev_snapshot, cbev_restore) without a GPU: the entry points reject a null handle before any CUDA
call, cbev_snapshot_info has the same layout in C (g++ probe of include/cbev.h) and in the ctypes mirror, and the
Python front end checks host index arrays before it touches the device."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIELDS = ("engine_token", "pool_epoch", "retreat_slots", "row_bytes", "n_rows", "reserved")


def test_new_entry_points_reject_a_null_handle():
    from carlabev_env_b200 import engine

    lib = engine.load_library()
    info = engine.CbevSnapshotInfo()
    buf = (C.c_uint8 * 64)()
    assert lib.cbev_snapshot_row_bytes(None) == -1
    assert lib.cbev_snapshot(None, None, 1, C.addressof(buf), 64, C.byref(info), None) == 1
    assert b"null handle" in lib.cbev_last_error()
    assert lib.cbev_restore(None, C.byref(info), C.addressof(buf), None, None, 1, None) == 1
    assert b"null handle" in lib.cbev_last_error()


def test_header_declares_snapshot_entry_points():
    from carlabev_env_b200 import engine

    header = open(os.path.join(ROOT, "include", "cbev.h")).read()
    for name in ("cbev_snapshot_row_bytes", "cbev_snapshot", "cbev_restore"):
        assert re.search(rf"\b{name}\(", header) and name in engine.EXPORTS, name
    # the struct name is never followed by "(": the export check collects every `cbev_...(` of the header
    assert not re.search(r"cbev_snapshot_info\s*\(", header)
    assert "} cbev_snapshot_info;" in header


def test_snapshot_info_layout_matches_ctypes(tmp_path):
    from carlabev_env_b200 import engine

    src = tmp_path / "probe.cpp"
    body = "\n".join(f'  printf("%zu\\n", offsetof(cbev_snapshot_info, {f}));' for f in FIELDS)
    src.write_text('#include <cstddef>\n#include <cstdio>\n#include "cbev.h"\nint main() {\n'
                   '  printf("%zu\\n", sizeof(cbev_snapshot_info));\n' + body + "\n  return 0;\n}\n")
    exe = tmp_path / "probe"
    subprocess.run(["g++", "-std=c++17", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    S = engine.CbevSnapshotInfo
    assert got == [C.sizeof(S)] + [getattr(S, f).offset for f in FIELDS]
    assert C.sizeof(S) == 32 and [f for f, _ in S._fields_] == list(FIELDS)


def _bare_engine(n):
    """An Engine shell with only what the host-side index checks read (no device, no library handle)."""
    import torch

    from carlabev_env_b200 import engine as E

    eng = E.Engine.__new__(E.Engine)
    eng.torch, eng.N, eng.device = torch, n, torch.device("cuda", 0)
    return eng


@pytest.mark.parametrize("idx,match", [
    ([0, 8], r"\[0, 8\)"),
    ([-1], r"\[0, 8\)"),
    ([], "non-empty"),
    ([[0, 1]], "1-D"),
    ([0.5], "integer"),
])
def test_host_indices_are_range_checked(idx, match):
    eng = _bare_engine(8)
    with pytest.raises(ValueError, match=match):
        eng._index(np.asarray(idx), 8, "env_ids", unique=True)


def test_host_restore_targets_must_be_distinct():
    eng = _bare_engine(8)
    with pytest.raises(ValueError, match="more than once"):
        eng._index([1, 2, 1], 8, "env_ids", unique=True)


def test_restore_takes_a_snapshot_object():
    eng = _bare_engine(8)
    with pytest.raises(TypeError, match="EnvSnapshot"):
        eng.restore(object())
