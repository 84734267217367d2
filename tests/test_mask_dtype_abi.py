"""uint8 semantic masks (CBEV_OBS_SEMANTIC_U8, mask_dtype="uint8") without a GPU: the C ABI validates the new
observation mode before any CUDA call, and the Python front ends reject what the option cannot mean."""
import ctypes

import pytest

OBS_SEMANTIC_U8 = 3  # include/cbev.h


def _cfg(**kw):
    from carlabev_env_b200 import engine

    cfg = engine.CbevConfig()
    cfg.num_envs, cfg.fov_size, cfg.anchor_x_frac, cfg.anchor_y_frac = 4, 128, 0.5, 0.5
    cfg.obs_h, cfg.obs_w, cfg.obs_mode, cfg.mask_mode = 96, 96, OBS_SEMANTIC_U8, engine.MASK_MODES["6-class"]
    cfg.frame_stack, cfg.ring_slots, cfg.n_discrete = 4, 8, 1
    for k, v in kw.items():
        setattr(cfg, k, v)
    return cfg


def _create(cfg):
    from carlabev_env_b200 import engine

    lib = engine.load_library()
    h = ctypes.c_void_p()
    rc = lib.cbev_create(ctypes.byref(cfg), ctypes.byref(h))
    return rc, lib.cbev_last_error().decode()


def test_header_declares_the_uint8_mask_mode():
    import os
    import re

    from carlabev_env_b200 import engine
    from golden_util import ROOT

    header = open(os.path.join(ROOT, "include", "cbev.h")).read()
    assert int(re.search(r"#define CBEV_OBS_SEMANTIC_U8 (\d+)", header).group(1)) == engine.OBS_SEMANTIC_U8 == 3
    assert re.search(r"int cbev_fuse\(cbev_handle h, int32_t mode, void\* out_dev, void\* stream\);", header)


def test_uint8_masks_need_planes_of_whole_16_byte_stores():
    rc, msg = _create(_cfg(obs_h=90, obs_w=90))  # 8100 % 16 != 0 (fine for float32 masks: 8100 % 4 == 0)
    assert rc == 1 and "multiple of 16" in msg and "16-byte stores" in msg, msg


def test_uint8_masks_validate_the_mask_mode():
    rc, msg = _create(_cfg(mask_mode=6))
    assert rc == 1 and "bad mask_mode 6" in msg, msg
    rc, msg = _create(_cfg(mask_mode=-1))
    assert rc == 1 and "mask_mode" in msg, msg


def test_observation_modes_beyond_the_uint8_masks_are_rejected():
    rc, msg = _create(_cfg(obs_mode=4))
    assert rc == 1 and "bad obs_mode 4" in msg, msg


def test_engine_rejects_mask_dtype_it_cannot_honour():
    from carlabev_env_b200 import engine as E

    with pytest.raises(ValueError, match="mask_dtype"):
        E.Engine(4, obs_mode=E.OBS_SEMANTIC, mask_dtype="float16")
    for mode in (E.OBS_GRAY, E.OBS_RGB):
        with pytest.raises(ValueError, match="semantic"):
            E.Engine(4, obs_mode=mode, mask_dtype="uint8")
    with pytest.raises(ValueError, match="mask_dtype='uint8'"):
        E.Engine(4, obs_mode=E.OBS_SEMANTIC_U8)


def test_make_env_rejects_mask_dtype_it_cannot_honour():
    from carlabev_env_b200 import EnvConfig, RunConfig, make_env

    with pytest.raises(ValueError, match="semantic"):
        make_env(RunConfig(num_envs=2, env=EnvConfig(obs_mode="bev_rgb")), mask_dtype="uint8")
    with pytest.raises(ValueError, match="mask_dtype"):
        make_env(RunConfig(num_envs=2), mask_dtype="float16")
