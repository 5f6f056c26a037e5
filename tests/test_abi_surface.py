"""CPU only: libshipsim.so loads and exports every entry point include/shipsim.h declares; the ctypes mirror of
`shipsim_config` has the C layout; with no GPU every call fails loudly (there is no CPU fallback).
No compute call is made here."""
import ctypes as C
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "shipsim.h")


def _declared():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(shipsim_[a-z_0-9]+)\s*\(", src)))


def test_header_declares_what_the_binding_lists():
    from ship_sim_gym_b200 import _abi
    assert sorted(_abi.SYMBOLS) == _declared()


def test_library_exports_every_declared_symbol():
    from ship_sim_gym_b200 import _abi
    lib = _abi.load()
    for name in _declared():
        assert getattr(lib, name) is not None, name
    assert lib.shipsim_abi_version() == 4
    # the dynamic symbol table too (what a cgo / JNI / ctypes binder would resolve against)
    out = subprocess.run(["nm", "-D", "--defined-only", _abi.LIB_PATH], capture_output=True, text=True).stdout
    exported = set(re.findall(r"\bT (shipsim_[a-z_0-9]+)", out))
    assert set(_declared()) <= exported


def test_header_compiles_as_plain_c(tmp_path):
    """The boundary is a C ABI: the header must be consumable by a C compiler with no CUDA / C++ headers."""
    src = tmp_path / "t.c"
    src.write_text('#include "shipsim.h"\nint main(void){shipsim_config c; return (int)sizeof(c) == 0;}\n')
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-c", str(src),
                           "-o", str(tmp_path / "t.o")])


def test_config_struct_layout_and_reference_defaults(tmp_path):
    from ship_sim_gym_b200 import _abi
    cfg = _abi.default_config()
    assert cfg.struct_size == C.sizeof(_abi.Config)
    # sizeof as the C compiler sees it
    src = tmp_path / "s.c"
    src.write_text('#include <stdio.h>\n#include "shipsim.h"\nint main(void){printf("%zu", sizeof(shipsim_config)); return 0;}\n')
    exe = tmp_path / "s"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    assert int(subprocess.check_output([str(exe)])) == C.sizeof(_abi.Config)
    # reference defaults: config.py:14-24, models.py:29,87,107, game.py:82,274-275, ship_env.py:13
    assert (cfg.bounds_w, cfg.bounds_h) == (600.0, 600.0)
    assert cfg.dt == pytest.approx(1.0) and cfg.damping == pytest.approx(0.4)
    assert cfg.max_steps == 1000 and cfg.history == 2 and cfg.lidar_beams == 10
    assert cfg.lidar_spread_deg == 90.0 and cfg.lidar_distance == 100.0
    assert (cfg.ship_w, cfg.ship_h, cfg.mass, cfg.thrust) == (2.0, 3.0, 5.0, 100.0)
    assert cfg.goal_radius == 5.0 and cfg.step_penalty == pytest.approx(-0.01) and cfg.spawn_y == 25.0


def test_argument_errors_do_not_need_a_gpu():
    from ship_sim_gym_b200 import _abi
    lib = _abi.load()
    h = C.c_void_p()
    cfg = _abi.default_config()
    cfg.history = 0
    assert lib.shipsim_create(C.byref(cfg), 0, C.byref(h)) == -1       # ValueError on the Python side (ship_env.py:46-47)
    assert b"history_size" in lib.shipsim_last_error()
    with pytest.raises(ValueError):
        _abi.check(-1)
    cfg = _abi.default_config()
    cfg.struct_size = 4
    assert lib.shipsim_create(C.byref(cfg), 0, C.byref(h)) == -1
    # the ship and goal knobs are checked before any device is looked for
    nan, inf = float("nan"), float("inf")
    for field, bad in [("mass", 0.0), ("mass", -5.0), ("mass", nan), ("mass", inf), ("ship_w", 0.0), ("ship_w", -2.0),
                       ("ship_h", 0.0), ("ship_h", nan), ("ship_w", inf), ("goal_radius", -0.5), ("goal_radius", nan),
                       ("thrust", inf), ("thrust", nan), ("lidar_spread_deg", inf), ("lidar_spread_deg", nan),
                       ("spawn_y", nan), ("spawn_y", -inf), ("step_penalty", nan)]:
        cfg = _abi.default_config()
        setattr(cfg, field, bad)
        assert lib.shipsim_create(C.byref(cfg), 0, C.byref(h)) == -1, (field, bad)
        assert field.split("_")[0].encode() in lib.shipsim_last_error(), (field, lib.shipsim_last_error())
    assert lib.shipsim_step(None, None, 0, 1, None, None, None, None) == -1
    assert lib.shipsim_destroy(None) == 0


def test_no_cpu_fallback():
    """Without a usable sm_100 device the product refuses to construct an env (it never routes to the oracle)."""
    torch = pytest.importorskip("torch")
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from ship_sim_gym_b200 import _abi
    lib = _abi.load()
    h = C.c_void_p()
    cfg = _abi.default_config()
    assert lib.shipsim_create(C.byref(cfg), 0, C.byref(h)) == -2
    assert b"no CPU fallback" in lib.shipsim_last_error()
    from ship_sim_gym_b200 import BatchedShipEnv
    with pytest.raises(Exception):
        BatchedShipEnv(4)


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "ship_sim_gym_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", "Makefile")):
                txt = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(import|from)\s+oracle\b", txt, flags=re.M), f
                assert "libshipsim_oracle" not in txt, f
