"""The 50 bonus levels (babyai/levels/bonus_levels.py) against the REFERENCE ITSELF: the reference's unmodified level classes
on the gym_minigrid shim (Philox back-end), step by step against the host build of the kernel source (tests/hostemu) --
observation, direction, mission, reward, done, every grid cell, agent pose, carried object, step counters and the number
of RNG draws (oracle/compare_ref.py), recorded from the reference into tests/golden/ref_runs.npz (make_ref_golden.py).  The
C oracle does not cover these families: their checker is the reference's runs and the reference-generated traces under
tests/golden/bonus_*.npz, which the CUDA pool replays."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.normpath(os.path.join(os.path.dirname(os.path.abspath(__file__)), '..'))
for p in (ROOT, os.path.join(ROOT, 'oracle'), os.path.join(ROOT, 'tests', 'hostemu')):
    if p not in sys.path:
        sys.path.insert(0, p)
from babyai_b200.levels import BONUS_LEVELS, detokenize, level_spec  # noqa: E402
from common import replay_reference_runs  # noqa: E402


class _One(object):
    """a one-env host-build pool with the oracle's interface"""

    def __init__(self, level, seed):
        import hostemu
        self.p = hostemu.HostEmuPool(level_spec(level), 1, np.array([seed], dtype=np.uint64))

    direction = property(lambda self: self.p.direction)

    def reset(self):
        return self.p.reset()

    def step(self, a):
        return self.p.step(np.asarray(a, dtype=np.int8))

    def mission(self, i):
        return detokenize(self.p.tokens(i))

    def state(self, i):
        return self.p.state(i)


@pytest.mark.timeout(600)
@pytest.mark.parametrize('level', BONUS_LEVELS)
def test_bonus_level_equals_reference(level):
    """3 random-action runs and (where the reference's bot returns) one bot-driven run per level"""
    replay_reference_runs('bonus', level, make_pool=_One)
