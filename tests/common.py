"""Shared helpers for the parity tests: replay a golden trace / a random action
stream through any pool-like object (oracle, host emulation, CUDA pool)."""
import json
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')
CONFIG_LEVELS = ['GoToRedBall', 'GoToLocal', 'PickupLoc', 'GoTo', 'BossLevel']
GOLDEN_LEVELS = sorted(f[:-4] for f in os.listdir(GOLDEN) if f.endswith('.npz') and not f.startswith(('succ_', 'rgb_', 'done_', 'bonus_', 'ref_')))      # all 47 served levels (CPU replays)
# success-heavy reference traces (97 % bot actions, >= 50 successful episodes each; make_golden.py --success): 'succ_<Level>'
# reference traces generated with BABYAI_DONE_ACTIONS=1 (verifier.use_done_actions; make_golden.py --done-actions): 'done_<Level>'
DONE_GOLDENS = sorted(f[:-4] for f in os.listdir(GOLDEN) if f.endswith('.npz') and f.startswith('done_'))
# reference traces of the 50 bonus levels (babyai/levels/bonus_levels.py; make_golden.py --bonus): 'bonus_<Level>'
BONUS_GOLDENS = sorted(f[:-4] for f in os.listdir(GOLDEN) if f.endswith('.npz') and f.startswith('bonus_'))
SUCCESS_GOLDENS = sorted(f[:-4] for f in os.listdir(GOLDEN) if f.endswith('.npz') and f.startswith('succ_'))
# the traces the CUDA pool replays in the GPU suite (the other 26 files were added at the very end of round 1, after the
# last GPU visit: they are replayed by the oracle and by the host build of the kernel logic; GPU replay from round 2 on)
GOLDEN_LEVELS_GPU = ['BossLevel', 'BossLevelNoUnlock', 'GoTo', 'GoToLocal', 'GoToObjMazeS4R2', 'GoToOpen', 'GoToRedBall',
                     'GoToRedBallGrey', 'GoToSeq', 'MiniBossLevel', 'Open', 'Pickup', 'PickupLoc', 'PutNext', 'PutNextLocal',
                     'PutNextLocalS5N3', 'Synth', 'SynthSeq', 'UnblockPickup']


REFERENCE_RUNS = os.path.join(GOLDEN, 'ref_runs.npz')
BOT_HANGS = ('UnlockToUnlock', 'KeyInBox')                 # the reference's bot does not return on these (its search loops)


def reference_runs():
    """Every run of the reference's own level code that the step-by-step comparisons replay, as (group, level, arguments of
    compare_ref.record); tests/golden/make_ref_golden.py records them into ref_runs.npz."""
    from babyai_b200.levels import BONUS_LEVELS, ICLR19_LEVELS
    runs = [('config_random', lv, dict(seed=4000 + s, steps=150, policy='random', act_seed=s)) for lv in CONFIG_LEVELS for s in range(2)]
    runs += [('iclr_random', lv, dict(seed=7100 + 17 * s, steps=300, policy='random', act_seed=10 + s))
             for lv in sorted(ICLR19_LEVELS) for s in range(3)]
    runs += [('iclr_bot', lv, dict(seed=7300, steps=200, policy='bot', act_seed=3)) for lv in sorted(ICLR19_LEVELS)]
    runs += [('bot', lv, dict(seed=5000, steps=250, policy='bot', act_seed=1))
             for lv in ['GoToLocal', 'PickupLoc', 'BossLevel', 'SynthSeq', 'GoToImpUnlock', 'Unlock']]
    for lv in BONUS_LEVELS:
        # reset() of a *Carrying level hands back the pre-carry observation: the states differ until the first step
        flags = dict(state_at_reset=not lv.endswith('Carrying'), check_draws=False)
        runs += [('bonus', lv, dict(seed=300 + 7 * k, steps=160, policy='random', act_seed=k, **flags)) for k in range(3)]
        if lv not in BOT_HANGS:
            runs.append(('bonus', lv, dict(seed=900, steps=160, policy='bot', act_seed=5, **flags)))
    return runs


_recorded = {}


def replay_reference_runs(group, level, make_pool=None):
    """Replays the recorded reference runs of (group, level) on a one-env pool (compare_ref.replay); returns the number of
    episodes that ended."""
    import compare_ref
    if not _recorded:                       # the runs are stored end to end (make_ref_golden.py runs())
        z = np.load(REFERENCE_RUNS)
        a = np.concatenate([[0], np.cumsum(z['steps'])])
        c = np.concatenate([[0], np.cumsum((z['steps'] + compare_ref.EVERY - 1) // compare_ref.EVERY)])
        for i, key in enumerate(json.loads(str(z['keys']))):
            _recorded[key] = z['actions'][a[i]:a[i + 1]], z['checks'][c[i]:c[i + 1]]
    runs = [kw for g, lv, kw in reference_runs() if (g, lv) == (group, level)]
    assert runs, (group, level)
    episodes = 0
    for kw in runs:
        actions, checks = _recorded[compare_ref.run_key(level, **kw)]
        flags = {k: kw[k] for k in ('state_at_reset', 'check_draws') if k in kw}
        episodes += compare_ref.replay(level, kw['seed'], actions, checks, make_pool=make_pool, **flags)
    return episodes


def load_golden(level):
    z = np.load(os.path.join(GOLDEN, level + '.npz'))
    d = {k: z[k] for k in z.files}
    d['missions'] = json.loads(str(d['missions']))
    return d


def replay_golden(level, make_pool, get_mission):
    """make_pool(level, n, seeds) -> object with reset() -> obs[n,7,7,3], step(a) -> (obs, reward, done),
    .direction; get_mission(pool, i) -> str.  All K traces are run as ONE pool of K envs."""
    g = load_golden(level)
    if level.startswith(('succ_', 'done_')):
        level = level[5:]
    elif level.startswith('bonus_'):
        level = level[6:]
    K, T = g['actions'].shape
    pool = make_pool(level, K, g['seeds'])
    obs = np.asarray(pool.reset())
    assert np.array_equal(obs.reshape(K, -1), g['obs0']), (level, 'reset obs')
    assert np.array_equal(np.asarray(pool.direction), g['dir0'])
    ep = [0] * K
    for i in range(K):
        assert get_mission(pool, i) == g['missions'][i][0]
    for t in range(T):
        obs, rew, done = pool.step(g['actions'][:, t])
        obs, rew, done = np.asarray(obs), np.asarray(rew), np.asarray(done)
        assert np.array_equal(done.astype(bool), g['done'][:, t].astype(bool)), (level, t, 'done')
        assert np.array_equal(rew.astype(np.float32).view(np.uint32), g['reward'][:, t].view(np.uint32)), (level, t, 'reward', rew, g['reward'][:, t])
        bad = np.nonzero((obs.reshape(K, -1) != g['obs'][:, t]).any(1))[0]
        assert len(bad) == 0, (level, t, 'obs differs for traces', bad)
        assert np.array_equal(np.asarray(pool.direction), g['direction'][:, t]), (level, t, 'direction')
        for i in np.nonzero(done)[0]:
            ep[i] += 1
            assert get_mission(pool, i) == g['missions'][i][ep[i]], (level, t, i)
    return int(g['done'].sum())


def compare_pools(a, b, n, steps, act_seed=0, mission_a=None, mission_b=None, state=True, check_draws=False, action_p=None):
    """Drive two pools with the same random actions (uniform, or distribution action_p); everything must be identical."""
    rng = np.random.RandomState(act_seed)
    oa, ob = np.asarray(a.reset()).copy(), np.asarray(b.reset()).copy()
    assert np.array_equal(oa, ob), 'reset obs'
    episodes = 0
    for t in range(steps):
        act = (rng.randint(0, 7, n) if action_p is None else rng.choice(7, size=n, p=action_p)).astype(np.int8)
        oa, ra, da = [np.asarray(x).copy() for x in a.step(act)]
        ob, rb, db = [np.asarray(x).copy() for x in b.step(act)]
        assert np.array_equal(da.astype(bool), db.astype(bool)), (t, 'done')
        assert np.array_equal(ra.view(np.uint32), rb.view(np.uint32)), (t, 'reward')
        bad = np.nonzero((oa != ob).reshape(n, -1).any(1))[0]
        assert len(bad) == 0, (t, 'obs', bad)
        assert np.array_equal(np.asarray(a.direction), np.asarray(b.direction)), (t, 'direction')
        episodes += int(da.astype(bool).sum())
        if state and (t % 7 == 0 or t == steps - 1):
            for i in range(n):
                g0, i0 = a.state(i)
                g1, i1 = b.state(i)
                assert np.array_equal(g0, g1), (t, i, 'grid')
                if not check_draws:
                    for k in ('draws', 'attempts'):
                        i0.pop(k), i1.pop(k)
                assert i0 == i1, (t, i, i0, i1)
                if mission_a is not None:
                    assert mission_a(a, i) == mission_b(b, i), (t, i)
    return episodes
