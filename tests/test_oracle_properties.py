"""CPU: what pins the float64 oracle BESIDES the golden trajectories (SURVEY.md §8c "what pins the restatement"):

1. the analytic known answers of SURVEY.md Appendix D (integrator, damping, thrust point, moment) -- derived from
   Chipmunk's documented cpBodyUpdatePosition / cpBodyUpdateVelocity / cpMomentForPoly, not measured on pymunk;
2. geometric self-consistency of the restated Chipmunk queries against independent brute-force formulations:
   segment-vs-convex-polygon (cpPolyShapeSegmentQuery) against Cyrus-Beck clipping, polygon-vs-polygon contact against
   exhaustive edge intersection / containment, point-to-polygon distance against the edge-by-edge minimum.
The oracle is test infrastructure; nothing here touches the CUDA path."""
import numpy as np
import pytest

import oracle
import parity
from helpers import source_constant
from oracle import cbind
from ship_sim_gym_b200 import ScenarioBank


def _env(speed, W=600.0, H=600.0, n=1, seed=0, **kw):
    bank = ScenarioBank.generate(4, (W, H), seed=seed).as_dict()
    env = oracle.OracleEnv(n, bank, W=W, H=H, speed=speed, **kw)
    env.reset(scen=[0] * n)
    return env


# ---------------------------------------------------------------------------------------------- Appendix D
APPENDIX_D = {          # SPEED -> y reported after steps 1.., straight thrust from rest (action 0 every step)
    1: [25.0, 25.2, 25.582489, 26.131488, 26.832419, 27.671979],
    10: [25.0, 45.0, 73.0, 104.2, 136.68, 169.672],
    30: [25.0, 205.0, 396.52, 588.77728],
    40: [25.0, 345.0, 673.192],
}


@pytest.mark.parametrize("speed", sorted(APPENDIX_D))
def test_straight_thrust_known_answers(speed):
    W = 1000.0 if speed >= 30 else 600.0
    env = _env(speed, W, W)
    ys = APPENDIX_D[speed]
    out = env.step(np.zeros((len(ys), 1), dtype=np.int32))
    obs = out["obs"][:, 0, 16:]
    assert np.allclose(obs[:, 1], ys, rtol=0, atol=2e-6)            # y
    assert np.all(obs[:, 0] == W / 2) and np.all(obs[:, 3] == 0.0)  # x stays exactly W/2, angle exactly 0 (no torque at rudder 0)
    dt, damp = 0.1 * speed, 0.4 ** (0.1 * speed)
    v = 0.0
    for _ in ys:
        v = v * damp + 20.0 * dt                                    # f/m = 100/5
    assert env.pose[0, 4] == pytest.approx(v, rel=1e-12) and env.pose[0, 3] == 0.0
    assert v < 20.0 * dt / (1.0 - damp)                             # below the terminal velocity of the table


def test_rudder_then_thrust_known_answers():
    env = _env(10)
    out = env.step(np.array([[1], [0], [0], [0], [0]], dtype=np.int32))
    obs = out["obs"][:, 0, 16:]
    assert list(obs[:, 2]) == [-5.0] * 5                            # rudder -5 after the single action 1
    # a rudder action alone produces no force or torque: the pose of step 1 is the spawn pose
    assert obs[0, 0] == 300.0 and obs[0, 1] == 25.0 and obs[0, 3] == 0.0
    # thrust at local point (-rudder, 0): torque = -100 * rudder = +500 about a moment of 3087.5
    assert np.allclose(obs[1:, 3], [0.0, 0.161943, 0.388664, 0.641296], atol=1e-6)
    assert env.pose[0, 5] == pytest.approx(0.262996, abs=1e-6)
    assert env.pose[0, 0] < 300.0                                   # positive angle = counter-clockwise: drift toward -x
    assert env.moment == pytest.approx(3087.5, rel=1e-12)
    assert cbind.moment_for_poly(5.0, env.ship_hull()) == pytest.approx(3087.5, rel=1e-12)


def test_noop_from_rest_and_spawn_observation():
    env = _env(10)
    obs0 = env.hist.copy()
    assert np.all(obs0[0, :16] == -1.0) and list(obs0[0, 16:20]) == [300.0, 25.0, 0.0, 0.0] and np.all(obs0[0, 22:] == -1.0)
    out = env.step(np.array([[1], [2]], dtype=np.int32))           # rudder -5, rudder back to 0: the hull never moves
    assert np.array_equal(env.pose[0], [300.0, 25.0, 0.0, 0.0, 0.0, 0.0])
    # at the spawn pose the lidar origin is (310, 47.5) and no ray reaches a bank of the default map: readings stay -1
    assert np.all(out["obs"][:, 0, 22:] == -1.0)
    assert np.all(out["reward"] == -0.01) and not out["done"].any()


def test_episode_length_cap_and_reward_priority():
    env = _env(1, max_steps=7)                                      # dt = 0.1: the ship barely moves in 7 steps
    out = env.step(np.full((7, 1), 1, dtype=np.int32))
    assert list(out["done"][:, 0]) == [0] * 6 + [1]                 # exactly MAX_STEPS steps (ship_env.py:131,152)
    assert np.all(out["reward"] == -0.01)


# ---------------------------------------------------------------------------------------------- geometry
def _random_convex(rng, n, cx, cy, r):
    ang = np.sort(rng.uniform(0, 2 * np.pi, n))
    rad = r * rng.uniform(0.6, 1.0, n)
    return cbind.convex_hull(np.stack([cx + rad * np.cos(ang), cy + rad * np.sin(ang)], 1))


def _inside(h, p, eps=0.0):
    e = np.roll(h, -1, axis=0) - h
    return np.all(e[:, 0] * (p[1] - h[:, 1]) - e[:, 1] * (p[0] - h[:, 0]) >= -eps)      # CCW: left of every edge


def _clip(h, a, b):
    """Cyrus-Beck: parameter range of a + t (b - a) inside the convex CCW polygon h, or None."""
    t0, t1 = 0.0, 1.0
    d = b - a
    for i in range(len(h)):
        p, q = h[i], h[(i + 1) % len(h)]
        nrm = np.array([q[1] - p[1], -(q[0] - p[0])])               # outward normal of a CCW edge
        num, den = nrm @ (a - p), nrm @ d
        if abs(den) < 1e-300:
            if num > 0:
                return None
            continue
        t = -num / den
        if den < 0:
            t0 = max(t0, t)
        else:
            t1 = min(t1, t)
    return (t0, t1) if t0 <= t1 else None


def test_segment_query_matches_cyrus_beck_clipping():
    rng = np.random.RandomState(0)
    n_hit = n_inside = n_miss = 0
    for _ in range(3000):
        h = _random_convex(rng, rng.randint(3, 13), 0.0, 0.0, 100.0)
        a = rng.uniform(-250, 250, 2)
        ang = rng.uniform(0, 2 * np.pi)
        b = a + 100.0 * np.array([np.cos(ang), np.sin(ang)])
        hit, point, alpha, margin = cbind.segment_query(h, a, b)
        if margin < 1e-6:
            continue                                               # grazing: either answer is legitimate
        if _inside(h, a):
            # cpShapeSegmentQuery: start inside the shape => reported at alpha 0 with `point` left at the segment END
            assert hit and alpha == 0.0 and np.allclose(point, b)
            n_inside += 1
            continue
        rng_t = _clip(h, a, b)
        if rng_t is None:
            assert not hit
            n_miss += 1
        else:
            assert hit and alpha == pytest.approx(rng_t[0], abs=1e-9)
            assert np.allclose(point, a + rng_t[0] * (b - a), atol=1e-7)
            n_hit += 1
    assert min(n_hit, n_inside, n_miss) > 100


def _seg_intersect(p, q, r, s):
    def orient(a, b, c):
        return (b[0] - a[0]) * (c[1] - a[1]) - (b[1] - a[1]) * (c[0] - a[0])
    o1, o2, o3, o4 = orient(p, q, r), orient(p, q, s), orient(r, s, p), orient(r, s, q)
    return (o1 > 0) != (o2 > 0) and (o3 > 0) != (o4 > 0)


def test_polygon_contact_matches_exhaustive_test():
    rng = np.random.RandomState(1)
    ship = np.array([[0, 0], [0, 30], [10, 45], [20, 30], [20, 0]], dtype=float)
    n_touch = n_apart = 0
    for _ in range(3000):
        bank = _random_convex(rng, rng.randint(3, 13), 0.0, 0.0, 120.0)
        th = rng.uniform(-np.pi, np.pi)
        R = np.array([[np.cos(th), -np.sin(th)], [np.sin(th), np.cos(th)]])
        hull = cbind.convex_hull(ship @ R.T + rng.uniform(-200, 200, 2))
        touch, sep = cbind.polys_touch(hull, bank)
        if abs(sep) < 1e-6:
            continue
        brute = any(_inside(bank, v) for v in hull) or any(_inside(hull, v) for v in bank) or any(
            _seg_intersect(hull[i], hull[(i + 1) % len(hull)], bank[j], bank[(j + 1) % len(bank)])
            for i in range(len(hull)) for j in range(len(bank)))
        assert touch == brute
        n_touch += touch
        n_apart += not touch
    assert min(n_touch, n_apart) > 300


def test_point_distance_matches_edgewise_minimum():
    rng = np.random.RandomState(2)
    for _ in range(2000):
        h = _random_convex(rng, rng.randint(3, 13), 0.0, 0.0, 50.0)
        p = rng.uniform(-100, 100, 2)
        best = np.inf
        for i in range(len(h)):
            a, b = h[i], h[(i + 1) % len(h)]
            t = np.clip((p - a) @ (b - a) / ((b - a) @ (b - a)), 0.0, 1.0)
            best = min(best, np.linalg.norm(p - (a + t * (b - a))))
        want = -best if _inside(h, p) else best                     # cpPolyShapePointQuery: negative inside
        assert cbind.poly_point_distance(h, p) == pytest.approx(want, abs=1e-9)


def test_scenario_picks_are_uniform_and_independent_of_neighbours():
    """The scenario an env plays next is an integer hash of (seed, global env id, episode) (the reference has no bank: it
    builds a level per reset, game.py:271-272).  What the batched env needs of it: uniform over the bank, no correlation
    between consecutive episodes of an env or between neighbouring envs, sensitive to every key word."""
    n_scen, n_env, n_ep = 64, 512, 256
    picks = np.array([[cbind.pick_scenario(12345, g, ep, n_scen) for ep in range(n_ep)] for g in range(n_env)])
    assert picks.min() == 0 and picks.max() == n_scen - 1
    counts = np.bincount(picks.ravel(), minlength=n_scen)
    expect = picks.size / n_scen
    chi2 = ((counts - expect) ** 2 / expect).sum()
    assert chi2 < 120, chi2                     # 63 degrees of freedom: mean 63, sd 11
    # consecutive episodes of an env, neighbouring envs at the same episode: pairs uniform over n_scen^2 -> equal with p = 1/n_scen
    same_next = (picks[:, 1:] == picks[:, :-1]).mean()
    same_nb = (picks[1:] == picks[:-1]).mean()
    assert abs(same_next - 1 / n_scen) < 0.004 and abs(same_nb - 1 / n_scen) < 0.004, (same_next, same_nb)
    # every word of the key matters: high seed word, high env-id word
    a = np.array([cbind.pick_scenario(12345, g, 3, 1 << 20) for g in range(64)])
    b = np.array([cbind.pick_scenario(12345 + (1 << 32), g, 3, 1 << 20) for g in range(64)])
    c = np.array([cbind.pick_scenario(12345, g + (1 << 32), 3, 1 << 20) for g in range(64)])
    assert (a != b).mean() > 0.95 and (a != c).mean() > 0.95


# ---------------------------------------------------------------------------------------------- the other knobs
# Appendix D holds the default ship only; the same closed forms hold for every mass, thrust and scale, and they pin the
# knob-dependent paths of the oracle before the GPU tests use it as the reference for those knobs.
def _fan_moment(mass, hull):
    """Moment about the body origin of a uniform polygon, summed over the triangles (0, v_i, v_i+1): each triangle's
    moment about its centroid, m (a^2 + b^2 + c^2) / 36, moved to the origin by the parallel-axis term m |centroid|^2."""
    v = np.asarray(hull, dtype=np.float64)
    w = np.roll(v, -1, axis=0)
    area = 0.5 * (v[:, 0] * w[:, 1] - v[:, 1] * w[:, 0])
    rho = mass / area.sum()
    sides = (v ** 2).sum(1) + (w ** 2).sum(1) + ((w - v) ** 2).sum(1)
    cen = (v + w) / 3.0
    m = rho * area
    return float((m * sides / 36.0 + m * (cen ** 2).sum(1)).sum())


@pytest.mark.parametrize("ship_w,ship_h,want", [(2.0, 3.0, 3087.5), (4.0, 5.0, 28112.5 / 3), (0.5, 0.5, None), (1.0, 7.0, None)])
def test_ship_moment_of_scaled_template(ship_w, ship_h, want):
    env = _env(10, ship_w=ship_w, ship_h=ship_h, mass=5.0)
    hull = env.ship_hull()
    tpl = parity.ship_hull(ship_w, ship_h)
    assert sorted(map(tuple, hull)) == sorted(map(tuple, tpl))         # the scaled template is its own convex hull
    assert env.moment == pytest.approx(_fan_moment(5.0, hull), rel=1e-12)
    if want is not None:
        assert env.moment == pytest.approx(want, rel=1e-12)
    env2 = _env(10, ship_w=ship_w, ship_h=ship_h, mass=12.5)
    assert env2.moment == pytest.approx(env.moment * 2.5, rel=1e-12)   # linear in the mass


@pytest.mark.parametrize("mass,thrust", [(5.0, 100.0), (1.5, 400.0), (50.0, 20.0), (0.25, 3.0)])
@pytest.mark.parametrize("speed", [1, 10])
def test_straight_thrust_follows_mass_and_thrust(mass, thrust, speed):
    W = 4000.0
    env = _env(speed, W, W, mass=mass, thrust=thrust)
    K = 5
    out = env.step(np.zeros((K, 1), dtype=np.int32))
    obs = out["obs"][:, 0, 16:]
    dt, damp = 0.1 * speed, 0.4 ** (0.1 * speed)
    v, y, ys = 0.0, 25.0, []
    for _ in range(K):
        y += v * dt                                                 # position first (cpBodyUpdatePosition), then velocity
        v = v * damp + (thrust / mass) * dt
        ys.append(y)
    assert np.allclose(obs[:, 1], ys, rtol=1e-12, atol=1e-9)
    assert np.all(obs[:, 0] == W / 2) and np.all(obs[:, 3] == 0.0)
    assert env.pose[0, 4] == pytest.approx(v, rel=1e-12) and env.pose[0, 3] == 0.0


@pytest.mark.parametrize("ship_w,ship_h,mass,thrust", [(2.0, 3.0, 5.0, 100.0), (4.0, 5.0, 5.0, 100.0), (0.5, 0.5, 1.5, 400.0),
                                                       (2.0, 3.0, 50.0, 20.0)])
def test_rudder_then_thrust_turns_by_torque_over_moment(ship_w, ship_h, mass, thrust):
    env = _env(10, 4000.0, 4000.0, ship_w=ship_w, ship_h=ship_h, mass=mass, thrust=thrust)
    out = env.step(np.array([[1], [0], [0], [0], [0]], dtype=np.int32))
    obs = out["obs"][:, 0, 16:]
    moment = _fan_moment(mass, parity.ship_hull(ship_w, ship_h))
    dt, damp = 1.0, 0.4
    w, a, angles = 0.0, 0.0, [0.0]
    for _ in range(4):
        a += w * dt
        w = w * damp + (5.0 * thrust / moment) * dt                 # torque = -rudder * F at rudder -5
        angles.append(a)
    assert np.allclose(obs[:, 3], angles, rtol=1e-10, atol=1e-12)
    assert env.pose[0, 5] == pytest.approx(w, rel=1e-10)


@pytest.mark.parametrize("W,H,spawn_y", [(900.0, 400.0, 25.0), (400.0, 1000.0, 25.0), (900.0, 400.0, 300.0), (1000.0, 1000.0, 300.0)])
def test_reset_observation_follows_bounds_and_spawn(W, H, spawn_y):
    bank = ScenarioBank.generate(4, (W, H), seed=1).as_dict()
    env = oracle.OracleEnv(3, bank, W=W, H=H, spawn_y=spawn_y)
    obs = env.reset(scen=[0, 1, 2])
    for e in range(3):
        g = bank["goals"][e]
        k = np.argmin(np.hypot(g[:, 0] - W / 2, g[:, 1] - spawn_y))
        want = [-1.0] * 16 + [W / 2, spawn_y, 0.0, 0.0, g[k, 0], g[k, 1]] + [-1.0] * 10
        assert list(obs[e]) == want


@pytest.mark.parametrize("penalty", [-0.01, -0.37, 0.0, 0.25])
def test_uneventful_step_returns_the_step_penalty(penalty):
    env = _env(10, step_penalty=penalty)
    out = env.step(np.array([[1], [2], [1]], dtype=np.int32))      # rudder only: the hull stays at the spawn pose
    assert np.all(out["reward"] == penalty) and not out["done"].any() and not out["flags"].any()
    assert env.ep_return[0] == pytest.approx(3 * penalty, abs=1e-15)


@pytest.mark.parametrize("radius", [0.5, 5.0, 40.0])
@pytest.mark.parametrize("ship", [(2.0, 3.0), (4.0, 5.0)])
def test_goal_taken_exactly_within_the_radius(radius, ship):
    W = H = 1000.0
    n = 600
    hull = parity.ship_hull(*ship)
    bank = ScenarioBank.generate(8, (W, H), seed=2).as_dict()
    rng = np.random.RandomState(3)
    pose, ints, lidar, goals, ret, delta = parity.goal_shell_states(rng, n, W, H, 8, hull=hull, radius=radius)
    env = oracle.OracleEnv(n, bank, W=W, H=H, goal_radius=radius, ship_w=ship[0], ship_h=ship[1], n_threads=4)
    parity.load_oracle_state(env, pose, ints, lidar, goals, ret)
    out = env.step(rng.randint(1, 3, n).astype(np.int32))           # rudder actions: the ship at rest stays put
    taken = (out["flags"] & oracle.FLAG_GOAL) != 0
    assert np.array_equal(taken, delta < 0)
    assert np.all(out["reward"][taken] == 1.0)
    assert np.allclose(out["margins"][:, parity.M_GOAL], np.abs(delta), rtol=0, atol=1e-9)


# ---------------------------------------------------------------------------------------------- reach-grid boundaries
@pytest.mark.parametrize("W,H", [(600.0, 600.0), (900.0, 400.0), (400.0, 1000.0), (4000.0, 4000.0)])
@pytest.mark.parametrize("ship", [(2.0, 3.0), (4.0, 5.0)])
def test_grid_boundary_states_straddle_the_cell_boundaries(W, H, ship):
    """The generator must put lidar origins within the stated ulps of the kernel's reach-grid boundaries: checked
    against the grid constants of the CUDA source, so that a change of the grid makes this fail instead of leaving the
    GPU tests that use the generator testing nothing in particular."""
    assert parity.GRID_N == source_constant("shipsim_device.cuh", r"constexpr int kGridN = (\d+);")
    assert parity.GRID_PAD == source_constant("shipsim_abi.cu", r"const double pad = ([0-9.]+);")
    hull = parity.ship_hull(*ship)
    rng = np.random.RandomState(0)
    n = 6000
    st, target = parity.grid_boundary_states(rng, n, W, H, 16, np.zeros((16, 5, 2)), hull=hull)
    pose = parity.f32_inputs(*st)[0]
    ox, oy = parity.lidar_origin(pose, hull)
    bnd = parity.grid_boundaries(W, H)
    beyond = np.zeros(n, dtype=bool)
    for a, (o, b, ext) in enumerate(((ox, bnd[0], W), (oy, bnd[1], H))):
        beyond |= (o < -parity.GRID_PAD) | (o > ext + parity.GRID_PAD)
        on = np.isin(target[:, a], parity.GRID_ULPS)
        i = np.abs(o[on, None] - b[None]).argmin(1)
        # the intended origin: the fp32 boundary moved by k ulps; the body coordinate that puts the origin there is
        # rounded to fp32, which may move it by half an ulp of that coordinate
        want = b[i].astype(np.float32)
        for k in (1, 2):
            for sgn in (1, -1):
                m = target[on, a] * sgn >= k
                want[m] = np.nextafter(want[m], np.float32(sgn * np.inf))
        slack = 0.5 * np.abs(np.spacing(pose[on, a].astype(np.float32))).astype(np.float64)
        assert np.all(np.abs(o[on] - want.astype(np.float64)) <= slack * (1 + 1e-9))
        assert set(np.unique(target[on, a])) == set(parity.GRID_ULPS)
        assert set(np.unique(i)) == set(range(parity.GRID_N + 1))      # every boundary, the outer ones included
        # at the inner boundaries the kernel's fp32 cell lookup lands on both sides
        o32 = np.float32(o[on])
        cell = parity.grid_cell(o32, ext)
        inner = (i > 0) & (i < parity.GRID_N)
        assert np.all((cell[inner] == i[inner]) | (cell[inner] == i[inner] - 1))
        assert (cell[inner] == i[inner]).sum() > 100 and (cell[inner] == i[inner] - 1).sum() > 100
        assert np.isin(cell, [0, parity.GRID_N - 1]).sum() > 20                # the unbounded border cells
    assert 0.08 < beyond.mean() < 0.2
