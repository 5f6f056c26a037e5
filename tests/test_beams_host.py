"""CPU: lidar fans other than the reference's 10 beams (LidarConfig.N_BEAMS, 1..32).

The float64 oracle has carried `n_beams` up to 32 all along; these tests pin that path -- fan geometry, a hand-computed
hit, the reset layout -- before the GPU tests compare the wide step kernel with it, and check the argument errors of
shipsim_create and the config snapshot.  Nothing here needs a GPU."""
import ctypes as C

import numpy as np
import pytest

import oracle
import parity
from helpers import fp32_bank, pack_bank


@pytest.mark.parametrize("spread", [90.0, 180.0, -120.0])
def test_twenty_beams_contain_the_ten_beam_fan(spread):
    """Ray 2i of a 20-beam fan has the angle of ray i of the 10-beam fan (delta halves, the start stays): over 32
    auto-reset steps from near-bank states its readings equal the 10-beam run's, and nothing else changes."""
    n, K = 512, 32
    bank = fp32_bank(16, 600, 600, seed=5)
    rng = np.random.RandomState(1)
    pose, ints, lidar, goals, ret = parity.f32_inputs(*parity.random_states(rng, n, 600, 600, 16, bank["goals"],
                                                                            near=(bank["hull_xy"], bank["hull_n"])))
    lidar20 = np.full((n, 20), -1.0)
    lidar20[:, 0::2] = lidar
    acts = rng.choice([0, 0, 1, 2], size=(K, n)).astype(np.int32)
    out = {}
    for nb, li in ((10, lidar), (20, lidar20)):
        orc = oracle.OracleEnv(n, bank, n_beams=nb, lidar_spread_deg=spread, auto_reset=True, seed=3)
        orc.reset()
        parity.load_oracle_state(orc, pose, ints, li, goals, ret, n_beams=nb)
        out[nb] = (orc.step(acts), orc.pose.copy(), orc.ints.copy())
    (r10, p10, i10), (r20, p20, i20) = out[10], out[20]
    o10, o20 = r10["obs"].reshape(K, n, 2, 16), r20["obs"].reshape(K, n, 2, 26)
    assert np.array_equal(o10[..., :6], o20[..., :6])
    assert np.abs(o20[..., 6::2] - o10[..., 6:]).max() <= 1e-9
    for key in ("reward", "done", "flags"):
        assert np.array_equal(r10[key], r20[key]), key
    assert np.array_equal(p10, p20) and np.array_equal(i10, i20)
    assert (o10[..., 6:] >= 0).mean() > 0.05               # the fans do hit the banks
    odd = o20[..., 7::2]
    assert ((odd >= 0) & (np.abs(odd - o20[..., 6::2]) > 1e-3)).any()    # and the rays between see something else


def test_single_ray_against_a_hand_computed_hit():
    """One ray at radians(90 - spread / 2) from the heading, from the lidar origin (body + half the hull's AABB), onto
    the lower face y = 260 of a wall bank: d = (260 - oy) / sin(angle)."""
    wall = np.array([[0.0, 260.0], [600.0, 260.0], [600.0, 320.0], [0.0, 320.0]])
    far = np.array([[0.0, -300.0], [600.0, -300.0], [600.0, -250.0], [0.0, -250.0]])
    goals = np.array([[100.0 * (i + 1), 500.0] for i in range(5)])
    bank = pack_bank([(wall, far)], [goals])
    spread = 60.0
    orc = oracle.OracleEnv(1, bank, n_beams=1, lidar_spread_deg=spread)
    orc.reset()
    x, y = 300.0, 200.0
    pose = np.array([[x, y, 0.0, 0.0, 0.0, 0.0]])
    ints = np.array([[0, 31, 0, 0, 0]], dtype=np.int32)
    parity.load_oracle_state(orc, pose, ints, np.array([[-1.0]]), goals.reshape(1, 10), np.zeros(1), n_beams=1)
    hx, hy = parity.lidar_origin_offset(np.zeros(1))
    ang = np.radians(90.0 - spread / 2.0)
    expect = (260.0 - (y + hy[0])) / np.sin(ang)
    assert 0 < expect < 100
    ref = orc.step(np.array([1], dtype=np.int32))         # rudder only: the pose does not move
    assert ref["obs"].shape == (1, 14)
    assert ref["obs"][0, -1] == pytest.approx(expect, rel=1e-12)
    assert ref["obs"][0, 7:13].tolist() == [x, y, -5.0, 0.0, goals[2, 0], goals[2, 1]]      # the nearest goal


@pytest.mark.parametrize("nb", [1, 7, 32])
def test_reset_observation_layout(nb):
    """ShipEnv.reset for n beams: [-1 x (6 + n) | x, y, 0, 0, gx, gy, -1 x n] (ship_env.py:180-184)."""
    bank = fp32_bank(4, 600, 600, seed=5)
    orc = oracle.OracleEnv(3, bank, n_beams=nb)
    obs = orc.reset()
    assert obs.shape == (3, 2 * (6 + nb))
    F = 6 + nb
    assert (obs[:, :F] == -1).all()
    assert (obs[:, F:F + 2] == [300.0, 25.0]).all()
    assert (obs[:, F + 2:F + 4] == 0).all()
    assert (obs[:, F + 4:F + 6] >= 0).all()
    assert (obs[:, F + 6:] == -1).all()


def test_snapshot_passes_the_beam_count_only_when_honoured():
    from ship_sim_gym_b200.config import EnvConfig, LidarConfig, snapshot

    class LC(LidarConfig):
        N_BEAMS = 32

    class EC(EnvConfig):
        LIDAR_CONFIG = LC

    assert snapshot(None, EC, honour_lidar_config=True)["lidar"]["N_BEAMS"] == 32
    assert snapshot(None, EC)["lidar"]["N_BEAMS"] == 10


def test_beam_count_errors_do_not_need_a_gpu():
    from ship_sim_gym_b200 import _abi
    lib = _abi.load()
    h = C.c_void_p()
    for bad in (0, -1, 33):
        cfg = _abi.default_config()
        cfg.lidar_beams = bad
        rc = lib.shipsim_create(C.byref(cfg), 0, C.byref(h))
        assert rc == -1, bad
        assert b"lidar_beams" in lib.shipsim_last_error()
        with pytest.raises(ValueError, match="lidar_beams"):
            _abi.check(rc)
    cfg = _abi.default_config()
    cfg.lidar_beams = 16
    cfg.steps_in_flight = 8
    rc = lib.shipsim_create(C.byref(cfg), 0, C.byref(h))
    assert rc == -4
    assert b"steps_in_flight" in lib.shipsim_last_error()
    with pytest.raises(NotImplementedError, match="steps_in_flight"):
        _abi.check(rc)
