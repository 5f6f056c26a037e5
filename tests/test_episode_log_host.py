"""CPU only: the host-side pieces of the episode log -- the header's record layout against the binding's constants, the
record -> dict conversion of BatchedShipEnv.episodes(), the HISTORY_SIZE > 2 row and terminal-row assembly and the
record -> info-dict conversion of ShipVecEnv(episode_info=True) -- on hand-made record tensors."""
import os
import re

import numpy as np
import pytest

torch = pytest.importorskip("torch")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _enum_values(names):
    src = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "shipsim.h")).read(), flags=re.S)
    vals, nxt = {}, 0
    for body in re.findall(r"enum\s*\{(.*?)\}", src, flags=re.S):
        nxt = 0
        for item in body.split(","):
            item = item.strip()
            if not item:
                continue
            m = re.match(r"(\w+)\s*(?:=\s*(\d+))?$", item)
            nxt = int(m.group(2)) if m.group(2) else nxt
            vals[m.group(1)] = nxt
            nxt += 1
    return {n: vals[n] for n in names}


def test_header_record_layout_matches_the_binding():
    from ship_sim_gym_b200 import _abi
    cols = ["K", "ENV", "LENGTH", "RETURN", "END", "SCENARIO", "EPISODE", "CALL"]
    v = _enum_values(["SHIPSIM_EP_" + c for c in cols])
    assert [v["SHIPSIM_EP_" + c] for c in cols] == [getattr(_abi, "EP_" + c) for c in cols] == list(range(8))
    ends = ["COLLISION", "ALL_GOALS", "OOB", "TIMEOUT", "GOAL"]
    v = _enum_values(["SHIPSIM_END_" + c for c in ends])
    assert [v["SHIPSIM_END_" + c] for c in ends] == [getattr(_abi, "END_" + c) for c in ends] == [1, 2, 4, 8, 16]
    assert "#define SHIPSIM_EPISODE_META 8" in open(os.path.join(ROOT, "include", "shipsim.h")).read()
    assert _abi.EPISODE_META == 8


def _records():
    from ship_sim_gym_b200 import _abi
    # (k, env, length, return, end, scenario, episode, call), deliberately out of order
    recs = [(3, 5, 12, 1.5, _abi.END_COLLISION, 7, 2, 1),
            (0, 9, 1000, -0.25, _abi.END_TIMEOUT | _abi.END_GOAL, 1, 0, 1),
            (3, 2, 40, 2.0, _abi.END_ALL_GOALS | _abi.END_GOAL, 3, 5, 1),
            (7, 0, 8, -1.0, _abi.END_OOB | _abi.END_TIMEOUT, 4, 1, 0)]
    meta = np.zeros((len(recs), 8), dtype=np.int32)
    for j, (k, e, ln, r, end, sc, ep, call) in enumerate(recs):
        meta[j] = (k, e, ln, np.float32(r).view(np.int32), end, sc, ep, call)
    rows = np.arange(len(recs) * 32, dtype=np.float32).reshape(len(recs), 32)
    return meta, rows


def test_episode_dict_sorts_and_decodes():
    from ship_sim_gym_b200.env import episode_dict
    meta, rows = _records()
    d = episode_dict(torch.from_numpy(meta), torch.from_numpy(rows), env_id_offset=100)
    assert d["call"].tolist() == [0, 1, 1, 1] and d["k"].tolist() == [7, 0, 3, 3] and d["env"].tolist() == [0, 9, 2, 5]
    assert d["global_env"].tolist() == [100, 109, 102, 105]
    assert d["return"].tolist() == [-1.0, -0.25, 2.0, 1.5] and d["return"].dtype == torch.float32
    assert d["length"].tolist() == [8, 1000, 40, 12]
    # truncated = the step cap alone (a goal taken on the last step does not change that)
    assert d["truncated"].tolist() == [False, True, False, False] and d["terminated"].tolist() == [True, False, True, True]
    assert d["oob"].tolist() == [True, False, False, False] and d["collision"].tolist() == [False, False, False, True]
    assert d["all_goals"].tolist() == [False, False, True, False] and d["goal"].tolist() == [False, True, True, False]
    assert d["scenario"].tolist() == [4, 1, 3, 7] and d["episode"].tolist() == [1, 0, 5, 2]
    assert torch.equal(d["terminal_obs"], torch.from_numpy(rows[[3, 1, 2, 0]]))


def test_long_history_terminal_rows():
    """H = 3: the env's row before the done step moved on by one frame, then the logged frame; -1 where that row had -1
    (frames older than the env's previous reset)."""
    from ship_sim_gym_b200.env import long_history_terminal_rows
    F, H, N, K = 16, 3, 4, 5
    prev = torch.arange(N * H * F, dtype=torch.float32).view(N, H * F)
    rows = 1000 + torch.arange(K * N * H * F, dtype=torch.float32).view(K, N, H * F)
    rows[2, 1, :F] = -1.0                                       # env 1 was reset at step 1: its row at step 2 starts with -1
    k = torch.tensor([0, 3, 4])
    env = torch.tensor([2, 1, 0])
    frame = -5.0 - torch.arange(3 * F, dtype=torch.float32).view(3, F)
    out = long_history_terminal_rows(prev, rows, k, env, frame)
    assert torch.equal(out[0], torch.cat([prev[2, F:], frame[0]]))
    assert torch.equal(out[1], torch.cat([rows[2, 1, F:], frame[1]]))
    assert torch.equal(out[2], torch.cat([rows[3, 0, F:], frame[2]]))
    out2 = long_history_terminal_rows(prev, rows, torch.tensor([3]), torch.tensor([1]), frame[:1])
    assert torch.equal(out2[0, F:2 * F], rows[2, 1, 2 * F:]) and bool((long_history_terminal_rows(
        prev, rows.clone().fill_(-1.0), torch.tensor([1]), torch.tensor([0]), frame[:1])[0, :2 * F] == -1.0).all())


@pytest.mark.parametrize("auto_reset", [False, True])
@pytest.mark.parametrize("H", [3, 4])
def test_long_history_rows_single_and_fused_steps(H, auto_reset):
    """HISTORY_SIZE > 2 rows at K = 1 follow the one-step rule: the previous row shifted by one frame, then the new frame;
    under auto-reset a done env's row is [-1 ... -1 | frame] instead.  One K-step call gives the rows of K one-step calls."""
    from ship_sim_gym_b200.env import long_history_rows
    F, N, K = 16, 8, 24
    g = torch.Generator().manual_seed(10 * H + auto_reset)
    prev = torch.rand(N, H * F, generator=g) * 600
    prev[:3, :F] = -1.0                                         # envs reset less than H steps ago
    frames = torch.rand(K, N, F, generator=g) * 600
    done = (torch.rand(K, N, generator=g) < 0.3).to(torch.uint8)
    assert ((done[1:] + done[:-1]) == 2).any()                  # done on consecutive steps: resets closer than H frames
    rows = long_history_rows(prev, frames, done, auto_reset)
    assert rows.shape == (K, N, H * F)
    row = prev
    for k in range(K):
        expect = torch.cat([row[:, F:], frames[k]], dim=1)
        if auto_reset:
            fresh = torch.full_like(expect, -1.0)
            fresh[:, -F:] = frames[k]
            expect = torch.where(done[k].bool()[:, None], fresh, expect)
        one = long_history_rows(row, frames[k:k + 1], done[k:k + 1], auto_reset)
        assert torch.equal(one[0], expect), k
        assert torch.equal(rows[k], expect), k
        row = one[0]


def test_vec_env_infos_from_records():
    from ship_sim_gym_b200.adapters import log_infos
    meta, rows = _records()
    base = [{} for _ in range(12)]
    infos = log_infos(base, meta, rows)
    assert all(infos[e] == {} for e in range(12) if e not in (0, 2, 5, 9))
    assert base == [{}] * 12                                    # the caller's list is not modified
    assert infos[9]["episode"] == {"r": -0.25, "l": 1000} and infos[9]["TimeLimit.truncated"] is True
    assert infos[0]["episode"] == {"r": -1.0, "l": 8} and infos[0]["TimeLimit.truncated"] is False
    assert infos[5]["episode"] == {"r": 1.5, "l": 12} and infos[2]["TimeLimit.truncated"] is False
    assert np.array_equal(infos[2]["terminal_observation"], rows[2])
    rows[2] = 0.0                                               # the info keeps its own copy of the row
    assert infos[2]["terminal_observation"][1] == 65.0
