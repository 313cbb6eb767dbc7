"""The C-ABI library loads and exports every entry point include/b200_gripper_sim.h declares; the CPU-only parts of the
boundary (model compiler, configuration defaults, error reporting) behave; the product refuses to run without a GPU."""
import ctypes as C
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "b200_gripper_sim.h")


def _declared():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return re.findall(r"GRS_API\s+[\w\s\*]+?\b(gr[spl]_\w+)\s*\(", src)


def test_library_exports_every_declared_symbol():
    from mujoco_rl_manipulate_unknown_objects_b200 import _native
    names = _declared()
    assert len(names) >= 35 and "grs_step" in names and "grp_forward" in names
    lib = C.CDLL(_native.lib_path())
    missing = [n for n in names if not hasattr(lib, n)]
    assert not missing, missing
    assert sorted(set(names)) == sorted(set(_native.SYMBOLS)), "python binding and header list different entry points"


def test_default_config_matches_reference_defaults():
    """config/base_config.py:29-43 of the reference."""
    from mujoco_rl_manipulate_unknown_objects_b200 import _native
    lib = _native.load()
    c = _native.GrsConfig()
    lib.grs_default_config(C.byref(c))
    assert (c.max_steps, c.time_horizon, c.include_roll, c.full_observation, c.im_reward, c.her_buffer, c.direction) == (400, 400, 1, 1, 0, 0, 0)
    assert (c.width, c.height) == (64, 64)
    assert np.allclose([c.pos_tolerance, c.grasp_tolerance, c.max_translation, c.max_rotation], [0.002, 0.03, 0.05, 0.15])


def test_compile_only_handle_has_no_device_state():
    from mujoco_rl_manipulate_unknown_objects_b200 import _native, compile_model
    cm = compile_model("/xmls/sugar_cube_env.xml")
    assert cm.sizes["nq"] == 14 and cm.sizes["nv"] == 13 and cm.sizes["nu"] == 7
    lib = _native.load()
    assert lib.grs_step(cm._h, None, None) != 0
    assert b"compile_only" in lib.grs_last_error() or b"null" in lib.grs_last_error()
    assert lib.grs_compile_only(b"/nonexistent/scene.xml") is None
    assert len(lib.grs_last_error()) > 0
    cm.close()


def test_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from mujoco_rl_manipulate_unknown_objects_b200 import GripperSim, make_config
    from mujoco_rl_manipulate_unknown_objects_b200.policy import GripperPolicy
    with pytest.raises(RuntimeError):
        GripperSim(make_config(sim_env="/xmls/sugar_cube_env.xml"), num_envs=2)
    with pytest.raises(RuntimeError):
        GripperPolicy(max_envs=2)
    from mujoco_rl_manipulate_unknown_objects_b200 import _native
    lib = _native.load()
    assert lib.grs_create(b"x.xml", 2, None, 0) is None and b"CUDA" in lib.grs_last_error()
    assert lib.grp_create(2, 5, 64, 64, 6, 0) is None and b"CUDA" in lib.grp_last_error()


def test_create_refuses_observations_larger_than_one_tile():
    """The observation is rasterised as one 64 x 64 tile: a larger width or height is refused by the configuration checks,
    before the device is looked at (so with or without a GPU)."""
    from mujoco_rl_manipulate_unknown_objects_b200 import _native
    lib = _native.load()
    for w, h in ((65, 64), (64, 65), (0, 64)):
        c = _native.GrsConfig()
        lib.grs_default_config(C.byref(c))
        c.width, c.height = w, h
        assert lib.grs_create(b"/xmls/sugar_cube_env.xml", 2, C.byref(c), 0) is None
        assert b"observation size must be within 1..64" in lib.grs_last_error(), lib.grs_last_error()


def test_config_struct_layout_is_the_same_in_header_binding_and_integration_stub():
    """grs_config is passed by pointer: the header, the package's ctypes binding and the stub shown in INTEGRATION.md must list the
    same fields in the same order with the same types, and the defaults of the trailing (non-reference) fields must be neutral."""
    from mujoco_rl_manipulate_unknown_objects_b200 import _native
    src = re.sub(r"/\*.*?\*/", "", open(HEADER).read(), flags=re.S)
    body = re.search(r"typedef struct grs_config \{(.*?)\} grs_config;", src, flags=re.S).group(1)
    header = []
    for decl in body.split(";"):
        decl = decl.strip()
        if not decl:
            continue
        ctype, names = decl.split(None, 1)
        header += [(n.strip(), ctype) for n in names.split(",")]
    ctype_of = {C.c_int32: "int32_t", C.c_float: "float", C.c_uint32: "uint32_t"}
    binding = [(n, ctype_of[t]) for n, t in _native.GrsConfig._fields_]
    assert header == binding
    assert C.sizeof(_native.GrsConfig) == 4 * len(header)
    stub = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    stub = stub[stub.index("class GrsConfig(C.Structure)"):stub.index("lib.grs_create.restype")]
    pos = [stub.index('"%s"' % n) for n, _ in header]  # every field named, in declaration order
    assert pos == sorted(pos)
    lib = _native.load()
    c = _native.GrsConfig()
    lib.grs_default_config(C.byref(c))
    assert (c.reset_noise_xy, c.reset_noise_yaw, c.seed) == (0.0, 0.0, 0)  # the reference's deterministic reset


def test_info_record_layout_matches_the_header():
    """The packed per-environment step record: the header's GRS_INFO_* enum (evaluated like a C compiler would) against the
    indices the Python layer uses to build `infos`."""
    from mujoco_rl_manipulate_unknown_objects_b200 import _native
    src = re.sub(r"/\*.*?\*/", "", open(HEADER).read(), flags=re.S)
    body = re.search(r"enum \{\s*(GRS_INFO_REWARD.*?)\};", src, flags=re.S).group(1)
    values, nxt = {}, 0
    for item in body.split(","):
        item = item.strip()
        if not item:
            continue
        name, _, val = item.partition("=")
        nxt = int(val) if val.strip() else nxt
        values[name.strip()[len("GRS_INFO_"):]] = nxt
        nxt += 1
    assert values == _native.INFO
    assert _native.INFO["STRIDE"] == 40 and _native.STATE_STRIDE == 64 and _native.RENDER_STATE_STRIDE == 96


def test_micro_benchmarks_compile_for_sm_100a(tmp_path):
    """tools/micro/*.cu (tcgen05.mma rate against N, per-SM bulk-copy streaming rate: the measurements DESIGN.md §3.3 quotes) build
    with the flags of the library; they only RUN on a B200."""
    import glob
    import shutil
    import subprocess
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    srcs = sorted(glob.glob(os.path.join(ROOT, "tools", "micro", "*.cu")))
    assert len(srcs) >= 2
    for src in srcs:
        r = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-c", "-o", str(tmp_path / "m.o"), src],
                           stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        assert r.returncode == 0, r.stdout
