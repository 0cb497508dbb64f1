"""The C-ABI shared library: loads, exports every symbol include/td_b200.h declares, validates arguments
and fails loudly without a GPU (no compute call is made here)."""
import ctypes as C
import os
import re

import pytest

from gym_td_b200 import engine as E
from gym_td_b200 import params

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    src = open(os.path.join(ROOT, "include", "td_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(td_[a-z_0-9]+)\s*\(", src)))


def test_header_symbols_are_exported():
    lib = E.lib()
    names = _declared()
    assert len(names) >= 20
    for n in names:
        assert hasattr(lib, n), "libtd_b200.so lacks %s" % n
    assert sorted(E.EXPORTS) == names
    assert lib.td_abi_version() == 3


def test_struct_sizes_match_header():
    assert C.sizeof(E.TdConfig) == 8 * 8 * 7 + 4 * 8 * 2 + 8 * 12 + 4 * 8
    assert C.sizeof(E.TdMap) == 4 * 8 + 2 * 64 * 64
    assert C.sizeof(E.TdStats) == 64
    assert E.HEADER_DTYPE.itemsize == 64


def test_ctypes_mirrors_have_the_headers_layout(tmp_path):
    """Size and every field offset of the ctypes structures, against what gcc sees in include/td_b200.h."""
    import subprocess
    pairs = {"td_config": E.TdConfig, "td_map": E.TdMap, "td_step_io": E.TdStepIO, "td_host_io": E.TdHostIO,
             "td_layout": E.TdLayout, "td_stats": E.TdStats}
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "td_b200.h"', 'int main(void) {']
    for cname, cls in pairs.items():
        lines.append('printf("%s size %%zu\\n", sizeof(%s));' % (cname, cname))
        for fname, _ in cls._fields_:
            lines.append('printf("%s %s %%zu\\n", offsetof(%s, %s));' % (cname, fname, cname, fname))
    records = {"td_env_header": E.HEADER_DTYPE, "td_tower_rec": E.TOWER_DTYPE, "td_enemy_rec": E.ENEMY_DTYPE}
    for cname, dt in records.items():
        lines.append('printf("%s size %%zu\\n", sizeof(%s));' % (cname, cname))
        for fname in dt.names:
            lines.append('printf("%s %s %%zu\\n", offsetof(%s, %s));' % (cname, fname, cname, fname))
    lines += ['return 0; }']
    src = tmp_path / "probe.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "probe"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)])
    got = {}
    for ln in subprocess.check_output([str(exe)], text=True).splitlines():
        struct, field, value = ln.split()
        got[(struct, field)] = int(value)
    for cname, cls in pairs.items():
        assert got[(cname, "size")] == C.sizeof(cls), cname
        for fname, _ in cls._fields_:
            assert got[(cname, fname)] == getattr(cls, fname).offset, (cname, fname)
    for cname, dt in records.items():                       # the numpy views of td_get_state blobs
        for fname in dt.names:
            assert got[(cname, fname)] == dt.fields[fname][1], (cname, fname)
    assert got[("td_env_header", "size")] == E.HEADER_DTYPE.itemsize == 64
    assert got[("td_tower_rec", "size")] == E.TOWER_DTYPE.itemsize == 16
    assert got[("td_enemy_rec", "size")] == E.ENEMY_DTYPE.itemsize == 24


def test_default_config_equals_reference_values():
    c = E.config_struct(params.Config())
    assert [list(r) for r in c.enemy_LP] == [[820, 1700], [2050, 3000], [6000, 8000], [8000, 12000]]
    assert [list(r) for r in c.tower_attack_interval][3] == [4.75, 4.75]
    assert (c.base_LP, c.max_cost, c.tower_distance, c.max_episode_steps, c.frozen_time) == (5, 100.0, 2, 1200, 2)
    cfg = params.Config()
    cfg.base_LP = None
    assert E.config_struct(cfg).base_LP == -1
    cfg.max_tower_lv = 2
    with pytest.raises(ValueError):
        E.config_struct(cfg)


@pytest.mark.parametrize("key,value", [("max_cost", 0), ("max_cost", -1.5), ("max_cost", float("nan")),
                                       ("enemy_cost", [[8, 8], [0, 15], [40, 40], [30, 30]]),
                                       ("enemy_cost", [[float("nan"), 8], [15, 15], [40, 40], [30, 30]])])
def test_config_with_a_zero_divisor_is_rejected(key, value):
    """Observation planes 11-12 divide by max_cost, 41-44 by enemy_cost[t][0]; the reference raises
    ZeroDivisionError on such a config, the engine refuses it up front."""
    cfg = params.Config()
    setattr(cfg, key, value)
    with pytest.raises(ValueError):
        E.config_struct(cfg)
    cfg = params.Config()
    cfg.enemy_cost = [[8, 0], [15, 0], [40, 0], [30, 0]]            # level 1 never divides
    cfg.max_cost = 1e-300
    assert E.config_struct(cfg).max_cost == 1e-300


def test_create_validates_and_reports():
    lib = E.lib()
    h = C.c_void_p()
    c = E.config_struct()
    assert lib.td_create(C.byref(c), 7, 10, 4, 0, C.byref(h)) == -1
    assert b"kind" in lib.td_last_error(None)
    assert lib.td_create(C.byref(c), 0, 3, 4, 0, C.byref(h)) == -1
    assert lib.td_create(C.byref(c), 0, 10, 0, 0, C.byref(h)) == -1


def test_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(E.TdError) as ei:
        E.Engine("def", 10, 4)
    assert ei.value.code == -2 and "no CPU fallback" in str(ei.value)
    import gym_td_b200
    with pytest.raises(E.TdError):
        gym_td_b200.make("TD-def-small-v0", seed=1)
    # the compressible-memory allocator is no exception: an error code and a message, no memory
    ptr = C.c_void_p(0x1234)
    assert E.lib().td_alloc_compressible(0, 1 << 20, C.byref(ptr), None) in (-2, -4) and not ptr.value
    assert E.lib().td_last_error(None)
    with pytest.raises(E.TdError):
        E.CompressibleBuffer(1 << 20, 0)


def _run_c_demo(tmp_path):
    import subprocess
    E.lib()                                                   # builds the library if needed
    cuda = "/usr/local/cuda"
    if not os.path.isdir(os.path.join(cuda, "include")):
        pytest.skip("CUDA toolkit headers not found")
    exe = tmp_path / "c_abi_demo"
    libdir = os.path.join(ROOT, "gym_td_b200")
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), "-I", os.path.join(cuda, "include"), "-o", str(exe),
                           os.path.join(ROOT, "examples", "c_abi_demo.c"), "-L", libdir, "-ltd_b200",
                           "-Wl,-rpath," + libdir, "-L", os.path.join(cuda, "lib64"), "-lcudart"])
    res = subprocess.run([str(exe), "256", "20"], capture_output=True, text=True, timeout=300)
    assert "ABI version 3" in res.stdout and "road(s)" in res.stdout
    return res


def test_plain_c_program_against_the_library(tmp_path):
    """examples/c_abi_demo.c: the boundary used from C alone.  Host-only entry points work everywhere; td_create
    reports TD_E_CUDA with a message on a box without a GPU (exit code 3) and the demo runs through on one."""
    res = _run_c_demo(tmp_path)
    assert res.returncode in (0, 3), res.stdout + res.stderr
    if res.returncode == 3:
        assert "no CPU fallback" in res.stdout
    else:
        assert "env-steps" in res.stdout


@pytest.mark.gpu
def test_plain_c_program_steps_envs_on_the_gpu(tmp_path):
    """The same C program on a GPU box: create, upload maps, reset, step, read statistics -- from C alone."""
    res = _run_c_demo(tmp_path)
    assert res.returncode == 0, res.stdout + res.stderr
    assert "env-steps" in res.stdout
