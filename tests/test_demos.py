"""The demo wire format (scripts/make_agent_demos.py:116, babyai/utils/demos.py:38-64): demos built from batched frozen-at-done
episodes must be what the reference's own one-env-at-a-time loop produces for the same seeds and actions (recorded in
tests/golden/ref_demos.npz by make_ref_golden.py), tuple for tuple after a pickle round trip."""
import json
import os
import pickle
import sys

import numpy as np
import pytest

ROOT = os.path.normpath(os.path.join(os.path.dirname(os.path.abspath(__file__)), '..'))


def _batched_episodes(level, seeds, acts):
    """N oracle envs stepped together without auto-reset (ManyEnvs flavour), the records DemoRecorder collects"""
    import oracle as orc
    n = len(seeds)
    pool = orc.OraclePool(level, n, np.array(seeds, dtype=np.uint64))
    obs = pool.reset().copy()
    missions = [pool.mission(i) for i in range(n)]
    T = acts.shape[0]
    imgs, dirs, dones, rews = [], [], [], []
    for t in range(T):
        imgs.append(obs.copy()); dirs.append(np.asarray(pool.direction).copy())
        o, r, d = pool.step(acts[t], autoreset=False)
        obs = o.copy(); dones.append(d.copy()); rews.append(r.copy())
    return missions, np.stack(imgs), np.stack(dirs), np.stack(dones), np.stack(rews)


DEMO_LEVELS = ['GoToLocal', 'PickupLoc', 'GoToObjMazeS4R2']


def demo_actions():
    """actions [T, n] and seeds of the demo comparison"""
    n, T, seed = 40, 150, 7000
    rng = np.random.RandomState(1)
    acts = rng.choice(7, size=(T, n), p=[0.15, 0.15, 0.45, 0.08, 0.05, 0.1, 0.02]).astype(np.int8)
    return acts, [seed + k for k in range(n)]


@pytest.mark.parametrize('level', DEMO_LEVELS)
def test_demos_equal_the_reference_loop(level):
    from babyai_b200.demos import episodes_to_demos
    acts, seeds = demo_actions()
    missions, imgs, dirs, dones, rews = _batched_episodes(level, seeds, acts)
    ours = pickle.loads(pickle.dumps(episodes_to_demos(missions, imgs, dirs, acts, dones, rews, pack_array=pickle.dumps)))
    # the reference's loop (make_agent_demos.generate_demos), one env at a time, same seeds, same action streams
    z = np.load(os.path.join(ROOT, 'tests', 'golden', 'ref_demos.npz'))
    theirs = json.loads(str(z[level + '.missions']))
    assert len(ours) == len(theirs) > 0
    t0 = 0
    for (mission, packed, directions, actions), want in zip(ours, theirs):
        t1 = t0 + len(actions)
        assert mission == want and np.array_equal(pickle.loads(packed), z[level + '.images'][t0:t1])
        assert list(directions) == z[level + '.directions'][t0:t1].tolist() and list(actions) == z[level + '.actions'][t0:t1].tolist()
        t0 = t1
    assert t0 == len(z[level + '.actions'])


def test_unfinished_and_failed_episodes_are_dropped():
    from babyai_b200.demos import episodes_to_demos
    T, n = 5, 3
    imgs = np.zeros((T, n, 7, 7, 3), np.uint8)
    done = np.zeros((T, n), bool); rew = np.zeros((T, n), np.float32)
    done[2, 0] = True; rew[2, 0] = 0.5                      # success after 3 steps
    done[4, 1] = True                                       # timed out: reward 0
    demos = episodes_to_demos(['a', 'b', 'c'], imgs, np.zeros((T, n), np.int8), np.ones((T, n), np.int8), done, rew, pack_array=pickle.dumps)
    assert len(demos) == 1 and demos[0][0] == 'a' and demos[0][3] == [1, 1, 1] and pickle.loads(demos[0][1]).shape == (3, 7, 7, 3)
    assert len(episodes_to_demos(['a', 'b', 'c'], imgs, np.zeros((T, n), np.int8), np.ones((T, n), np.int8), done, rew,
                                 pack_array=pickle.dumps, successful_only=False)) == 2


@pytest.mark.gpu
def test_demo_recorder_on_the_gpu():
    """DemoRecorder (pool in ManyEnvs mode, batched policy) == the same episodes through the oracle"""
    import torch
    from babyai_b200.demos import DemoRecorder
    n, seed = 64, 4200
    rec = DemoRecorder('GoToLocal', n, pack_array=pickle.dumps)
    g = torch.Generator(device='cuda').manual_seed(0)
    stream = []

    def policy(image, direction, tokens):
        a = torch.randint(0, 7, (n,), device='cuda', generator=g, dtype=torch.int8)
        a = torch.where(a >= 3, torch.full_like(a, 2), a)          # left / right / forward: GoTo missions succeed by wandering
        stream.append(a.cpu().numpy())
        return a
    demos = rec.record(policy, [seed + k for k in range(n)], max_steps=70)
    acts = np.stack(stream)
    missions, imgs, dirs, dones, rews = _batched_episodes('GoToLocal', [seed + k for k in range(n)], acts)
    from babyai_b200.demos import episodes_to_demos
    want = episodes_to_demos(missions, imgs, dirs, acts, dones, rews, pack_array=pickle.dumps)
    assert len(demos) == len(want) > 5
    for a, b in zip(demos, want):
        assert a[0] == b[0] and a[2] == b[2] and a[3] == b[3] and np.array_equal(pickle.loads(a[1]), pickle.loads(b[1]))
