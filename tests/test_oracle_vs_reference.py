"""Pins the C oracle against the reference itself: runs of the reference's
unmodified babyai.levels (levelgen.py, verifier.py, iclr19_levels.py) executing
on the clean-room gym_minigrid shim, compared step by step (obs, reward, done,
direction, mission, full grid, agent pose, carried object, step counters and the
number of RNG draws).  The reference's runs are recorded in
tests/golden/ref_runs.npz and ref_place_agent_hang.npz (make_ref_golden.py);
the tests marked `reference` run the reference's own code and need its tree."""
import json
import os

import numpy as np
import pytest

from common import CONFIG_LEVELS, GOLDEN, replay_reference_runs


@pytest.mark.parametrize('level', CONFIG_LEVELS)
def test_random_policy(level):
    replay_reference_runs('config_random', level)


def _iclr_levels():
    from babyai_b200.levels import ICLR19_LEVELS
    return sorted(ICLR19_LEVELS)


@pytest.mark.parametrize('level', _iclr_levels())
def test_random_policy_every_iclr_level(level):
    """every served ICLR-19 level, 3 seeds x 300 random steps (several episodes on the single-room levels, resets included):
    the CI-length slice of oracle/soak_ref.py (profiles/r02_soak_ref.log has the long run)"""
    replay_reference_runs('iclr_random', level)


@pytest.mark.parametrize('level', _iclr_levels())
def test_bot_policy_every_iclr_level(level):
    """... and the reference bot driving both sides (the success / reward path of every instruction kind)"""
    replay_reference_runs('iclr_bot', level)


@pytest.mark.parametrize('level', ['GoToLocal', 'PickupLoc', 'BossLevel', 'SynthSeq', 'GoToImpUnlock', 'Unlock'])
def test_bot_policy(level):
    eps = replay_reference_runs('bot', level)
    assert eps >= 0


@pytest.mark.reference
def test_reference_level_test_on_shim():
    """A slice of the reference's own test (levelgen.py:496-541) on the shim: determinism per seed."""
    import refenv
    refenv.setup('mt')
    from babyai.levels import level_dict
    for name in CONFIG_LEVELS:
        m0, m1 = level_dict[name](seed=0), level_dict[name](seed=0)
        assert m0.grid == m1.grid and m0.surface == m1.surface
        assert m0.reset()['mission'] == m0.surface


@pytest.mark.reference
def test_bot_solves_config_levels():
    import selfcheck_bot
    assert selfcheck_bot.run(CONFIG_LEVELS, 3, 'philox')


def test_reference_place_agent_hang_is_rejected():
    """RoomGrid.place_agent loops `while True` until the cell in front of the agent is empty or a wall
    (gym_minigrid/roomgrid.py place_agent).  MiniBossLevel, seed 698: the 57th level picks a 3x3 room whose two empty
    cells face objects / doors in all four headings, so the reference never returns (make_ref_golden.py records the 56
    levels before it and the grid it is stuck on).  The oracle (and the kernels) reject that level instead: same levels
    up to there, then the oracle carries on."""
    import oracle as orc
    z = np.load(os.path.join(GOLDEN, 'ref_place_agent_hang.npz'))
    missions = json.loads(str(z['missions']))
    pool = orc.OraclePool('MiniBossLevel', 1, np.array([698], dtype=np.uint64))
    assert len(missions) == len(z['obs']) == 56
    for k in range(56):
        oo = pool.reset()
        assert np.array_equal(np.asarray(oo)[0].reshape(7, 7, 3), z['obs'][k]), k
        assert pool.mission(0) == missions[k]
    # the room the reference is stuck in: no empty cell with an empty / wall cell in front of it
    grid = z['hung_grid']                                  # Grid.encode(): [x, y, (type, colour, state)]
    stuck = []
    for (i, j), top, size in zip(z['room_ij'], z['room_top'], z['room_size']):
        ok = False
        for y in range(top[1] + 1, top[1] + size[1] - 1):
            for x in range(top[0] + 1, top[0] + size[0] - 1):
                if grid[x, y, 0] != 1:                     # not an empty cell
                    continue
                for dx, dy in ((1, 0), (0, 1), (-1, 0), (0, -1)):
                    ok = ok or grid[x + dx, y + dy, 0] in (1, 2)         # empty or wall
        if not ok:
            stuck.append((i, j))
    assert stuck, 'expected a room without any admissible agent pose'
    pool.reset()        # returns: the oracle rejected the unsatisfiable level
    assert pool.state(0)[1]['attempts'] >= 58
