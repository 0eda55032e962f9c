"""The step-based env path without a GPU: the C ABI of fg_env_step (struct layout, argument validation before any CUDA
call), the resource usage of every k_env_step instantiation, and the input checks of BaseReacherEnv.step()."""
import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "fancy_gym_b200.h")


def test_env_step_struct_layout_matches_ctypes(tmp_path):
    from fancy_gym_b200 import _lib
    structs = {"fg_env_step_cfg": _lib.FgEnvStepCfg, "fg_env_step_io": _lib.FgEnvStepIO}
    lines = ['#include <stdio.h>', '#include <stddef.h>', f'#include "{HEADER}"', 'int main(void){']
    for name, cls in structs.items():
        lines.append(f'printf("{name} %zu\\n", sizeof({name}));')
        lines += [f'printf("{name}.{f} %zu\\n", offsetof({name}, {f}));' for f, _ in cls._fields_]
    lines += ['return 0;}']
    prog = tmp_path / "layout.c"
    prog.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-pedantic", str(prog), "-o", str(exe)], check=True)
    out = dict(line.split() for line in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines())
    for name, cls in structs.items():
        assert int(out[name]) == C.sizeof(cls), name
        for f, _ in cls._fields_:
            assert int(out[f"{name}.{f}"]) == getattr(cls, f).offset, (name, f)


def _valid_args(B=0):
    """a configuration that passes validation; the pointers are never dereferenced (every call below returns before a
    launch: B == 0 or one argument is invalid)"""
    from fancy_gym_b200 import _lib
    cfg = _lib.FgEnvStepCfg()
    cfg.struct_size = C.sizeof(_lib.FgEnvStepCfg)
    cfg.env_kind, cfg.n_dof, cfg.max_episode_steps, cfg.dt = _lib.ENV_HOLE_REACHER, 5, 200, 0.01
    io = _lib.FgEnvStepIO()
    io.struct_size = C.sizeof(_lib.FgEnvStepIO)
    for i, f in enumerate(("action", "q", "v", "steps", "done", "ctx", "latch", "obs", "reward", "flag_bytes", "info")):
        setattr(io, f, 0x10000 + 0x1000 * i)
    return cfg, io


def _call(cfg, io, B):
    from fancy_gym_b200 import _lib
    return _lib.lib.fg_env_step(C.byref(cfg), C.byref(io), B, None)


def test_env_step_validates_before_touching_cuda():
    from fancy_gym_b200 import _lib
    cfg, io = _valid_args()
    assert _call(cfg, io, 0) == _lib.OK                       # nothing to do: no launch

    cfg, io = _valid_args()
    cfg.struct_size = 3
    assert _call(cfg, io, 16) == _lib.ERR_INVALID and b"struct_size" in _lib.lib.fg_last_error()
    cfg, io = _valid_args()
    io.struct_size = C.sizeof(_lib.FgEnvStepIO) + 8
    assert _call(cfg, io, 16) == _lib.ERR_INVALID and b"struct_size" in _lib.lib.fg_last_error()

    cfg, io = _valid_args()
    cfg.env_kind = _lib.ENV_TOY
    assert _call(cfg, io, 16) == _lib.ERR_UNSUPPORTED
    with pytest.raises(NotImplementedError):
        _lib.check(_call(cfg, io, 16))
    cfg.env_kind = 7
    assert _call(cfg, io, 16) == _lib.ERR_INVALID

    for n in (-1, 0, 1, 8, 9):
        cfg, io = _valid_args()
        cfg.n_dof = n
        assert _call(cfg, io, 16) == _lib.ERR_UNSUPPORTED, n

    cfg, io = _valid_args()
    assert _call(cfg, io, -1) == _lib.ERR_INVALID and b"negative" in _lib.lib.fg_last_error()

    for f in ("action", "q", "v", "steps", "done", "ctx", "obs", "reward", "flag_bytes", "info"):
        cfg, io = _valid_args()
        setattr(io, f, None)
        assert _call(cfg, io, 16) == _lib.ERR_INVALID and b"NULL" in _lib.lib.fg_last_error(), f
    cfg, io = _valid_args()                                   # the latch is needed by the "unbounded" reward only
    cfg.rew_fct, io.latch = 2, None
    assert _call(cfg, io, 16) == _lib.ERR_INVALID
    cfg.rew_fct = 3
    assert _call(cfg, io, 16) == _lib.ERR_INVALID
    assert _lib.lib.fg_env_step(None, C.byref(io), 16, None) == _lib.ERR_INVALID


def test_env_step_kernels_do_not_spill():
    """every k_env_step instantiation (3 envs x 2..7 links x float32 / float64 actions) keeps its state in registers"""
    from fancy_gym_b200 import _lib
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    out = subprocess.run([cuobjdump, "--dump-resource-usage", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    usage, name = {}, None
    for line in out.splitlines():
        m = re.search(r"Function (\S+):", line)
        if m:
            name = m.group(1)
        m = re.search(r"REG:(\d+).*LOCAL:(\d+)", line)
        if m and name and "k_env_step" in name:
            usage[name] = (int(m.group(1)), int(m.group(2)))
    assert len(usage) == 36, sorted(usage)
    assert all(local == 0 for _, local in usage.values()), usage
    assert all(reg <= 128 for reg, _ in usage.values()), usage


def _cpu_env(**kw):
    from fancy_gym_b200.envs.classic_control import HoleReacherEnv
    return HoleReacherEnv(5, num_envs=4, device="cpu", context_sampler="numpy", **kw)


def test_step_checks_its_input_before_any_launch():
    env = _cpu_env()
    with pytest.raises(RuntimeError, match="reset"):
        env.step(np.zeros((4, 5), np.float32))              # gymnasium's OrderEnforcing: reset first
    env.reset(seed=0)
    with pytest.raises(TypeError):
        env.step(np.zeros((4, 5), np.int64))
    with pytest.raises(TypeError):
        env.step(np.zeros((4, 5), np.float16))
    with pytest.raises(ValueError):
        env.step(np.zeros((4, 4), np.float32))
    with pytest.raises(ValueError):
        env.step(np.zeros(5, np.float32))                   # [n] only when num_envs == 1


def test_make_vec_routes_step_based_ids():
    import fancy_gym_b200 as fg
    from fancy_gym_b200.envs.registry import bb_env_constructor
    from fancy_gym_b200.utils.gym_compat import registry
    for name in ("HoleReacher-v0", "ViaPointReacher-v0", "SimpleReacher-v0", "LongSimpleReacher-v0"):
        assert registry[f"fancy/{name}"].entry_point is not bb_env_constructor
        assert registry[f"fancy_ProMP/{name}"].entry_point is bb_env_constructor
    assert fg.StepVectorEnv is not fg.BlackBoxVectorEnv
