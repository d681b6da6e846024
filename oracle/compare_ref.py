"""Step-by-step comparison of the C oracle (oracle/babyai_oracle.c) with the
reference's own BabyAI layer running on the gym_minigrid shim, Philox back-end.
TEST INFRASTRUCTURE ONLY.  compare() and record() run the reference and need its
tree (refenv.REFERENCE); replay() checks a pool against what record() stored and
needs nothing outside this repository.

Checked at reset and after every step: observation image bytes, direction,
mission string, reward (as float32), done, and the full hidden state: every
grid cell's (type, color, state), agent pose, carried object, step_count,
max_steps and the number of RNG draws consumed.  record() keeps the actions it
played and a running digest of those values every EVERY steps; replay() plays
the same actions on the pool and recomputes the digest from the pool's values.
"""
import hashlib
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import refenv  # noqa: E402
import oracle as orc  # noqa: E402

EVERY = 20                                 # steps per stored digest checkpoint


def ref_state(env):
    g = env.grid
    img = g.encode()                       # [x, y, 3]
    packed = (img[:, :, 0] | (img[:, :, 1] << 3) | (img[:, :, 2] << 6)).astype(np.uint8).T   # [y, x]
    car = 0
    if env.carrying is not None:
        t = env.carrying.encode()
        car = t[0] | (t[1] << 3) | (t[2] << 6)
    return packed, dict(agent_x=int(env.agent_pos[0]), agent_y=int(env.agent_pos[1]), agent_dir=int(env.agent_dir),
                        carrying=int(car), step_count=int(env.step_count), max_steps=int(env.max_steps),
                        draws=int(env.np_random.draws) & 0x7FFFFFFF)


def check_state(env, pool, tag, check_draws=True):
    g0, i0 = ref_state(env)
    g1, i1 = pool.state(0)
    i1 = dict(i1)
    i1.pop('attempts')
    if not check_draws:                    # (a pool that generates levels ahead has consumed more draws)
        i0.pop('draws'); i1.pop('draws')
    assert np.array_equal(g0, g1), (tag, 'grid', g0, g1)
    assert i0 == i1, (tag, i0, i1)


def _reference_run(level, seed, steps, policy, act_seed):
    """The reference's side of a comparison.  policy: 'random' | 'bot' (reference bot, 25% random perturbation).
    Yields (env, obs) after reset, then (env, action, obs, reward, done) after every step; obs is the observation after
    the auto-reset (penv.py:9-10) when done."""
    env = refenv.make_env(level, seed, 'philox')
    rng = np.random.RandomState(act_seed)
    obs = env.reset()
    yield env, obs
    bot = None
    if policy == 'bot':
        from babyai.bot import Bot
        bot = Bot(env)
    last = None
    for t in range(steps):
        if bot is not None and rng.rand() < 0.75:
            try:
                a = int(bot.replan(last))
            except Exception:
                a = int(rng.randint(0, 7))
                bot = None
        else:
            a = int(rng.randint(0, 7))
            if bot is not None:
                # the bot cannot recover from opened boxes / closed doors (eval_bot.py:131-139)
                fc = env.grid.get(*env.front_pos)
                if a == 5 and fc is not None and (fc.type == 'box' or (fc.type == 'door' and fc.is_open)):
                    a = 6
        last = a
        obs, reward, done, _ = env.step(a)
        if done:
            obs = env.reset()                    # penv.py:9-10
            if policy == 'bot':
                from babyai.bot import Bot
                bot = Bot(env)
                last = None
        yield env, a, obs, reward, done


def compare(level, seed, steps, policy='random', act_seed=0, verbose=False, make_pool=None, state_at_reset=True, check_draws=True):
    """Runs the reference and a pool side by side.  make_pool(level, seed) -> a one-env pool with the oracle's interface
    (default: the C oracle); the bonus levels are checked with the host build of the kernel source."""
    run = _reference_run(level, seed, steps, policy, act_seed)
    env, obs = next(run)
    pool = orc.OraclePool(level, 1, seeds=[seed]) if make_pool is None else make_pool(level, seed)
    o = pool.reset()
    assert np.array_equal(obs['image'], o[0]), (level, seed, 'reset obs')
    assert obs['mission'] == pool.mission(0), (obs['mission'], pool.mission(0))
    if state_at_reset:
        check_state(env, pool, (level, seed, 'reset'), check_draws)
    episodes = 0
    for t, (env, a, obs, reward, done) in enumerate(run):
        episodes += int(done)
        o, r, d = pool.step([a])
        tag = (level, seed, t, a)
        assert bool(d[0]) == bool(done), (tag, 'done', d[0], done)
        assert np.float32(reward) == r[0], (tag, 'reward', reward, r[0])
        assert np.array_equal(obs['image'], o[0]), (tag, 'obs')
        assert obs['direction'] == pool.direction[0], (tag, 'dir')
        assert obs['mission'] == pool.mission(0), (tag, obs['mission'], pool.mission(0))
        if state_at_reset or not done:
            check_state(env, pool, tag, check_draws)
    return episodes


def run_key(level, seed, steps, policy, act_seed, state_at_reset=True, check_draws=True):
    """name of a recorded run (what record() was called with)"""
    return '%s-%s-%d-%d-%d-%d%d' % (level, policy, seed, steps, act_seed, state_at_reset, check_draws)


def _fold(h, image, mission, state=None, check_draws=True, direction=None, reward=None, done=None):
    """adds the values compare() checks to the running digest h, in one fixed byte layout for both sides"""
    h.update(np.ascontiguousarray(image, dtype=np.uint8).tobytes())
    h.update(mission.encode() + b'\0')
    if done is not None:
        h.update(np.array([bool(done), int(direction)], np.int64).tobytes() + np.float32(reward).tobytes())
    if state is not None:
        grid, info = state
        info = {k: int(v) for k, v in info.items() if k != 'attempts' and (check_draws or k != 'draws')}
        h.update(np.array(grid.shape, np.int64).tobytes() + np.ascontiguousarray(grid, dtype=np.uint8).tobytes())
        h.update(json.dumps(sorted(info.items())).encode())


def record(level, seed, steps, policy='random', act_seed=0, state_at_reset=True, check_draws=True):
    """The reference's run of compare(): (actions uint8[steps], digest checkpoints uint64[ceil(steps / EVERY)])."""
    run = _reference_run(level, seed, steps, policy, act_seed)
    env, obs = next(run)
    h = hashlib.blake2b(digest_size=8)
    _fold(h, obs['image'], obs['mission'], ref_state(env) if state_at_reset else None, check_draws)
    actions, checks = [], []
    for t, (env, a, obs, reward, done) in enumerate(run):
        actions.append(a)
        _fold(h, obs['image'], obs['mission'], ref_state(env) if state_at_reset or not done else None, check_draws,
              obs['direction'], reward, done)
        if (t + 1) % EVERY == 0 or t == steps - 1:
            checks.append(h.digest())
    return np.array(actions, np.uint8), np.frombuffer(b''.join(checks), np.uint64).copy()


def replay(level, seed, actions, checks, make_pool=None, state_at_reset=True, check_draws=True):
    """Plays a recorded run on a pool (make_pool as in compare()) and checks it step for step against the reference's
    digests; returns the number of episodes that ended."""
    pool = orc.OraclePool(level, 1, seeds=[seed]) if make_pool is None else make_pool(level, seed)
    h = hashlib.blake2b(digest_size=8)
    o = pool.reset()
    _fold(h, o[0], pool.mission(0), pool.state(0) if state_at_reset else None, check_draws)
    episodes = 0
    for t, a in enumerate(actions):
        o, r, d = pool.step([int(a)])
        done = bool(d[0])
        episodes += int(done)
        _fold(h, o[0], pool.mission(0), pool.state(0) if state_at_reset or not done else None, check_draws,
              pool.direction[0], r[0], done)
        if (t + 1) % EVERY == 0 or t == len(actions) - 1:
            k = t // EVERY
            assert h.digest() == checks[k].tobytes(), (level, seed, 'differs from the reference within steps %d..%d'
                                                       % (k * EVERY, t))
    assert len(checks) == (len(actions) + EVERY - 1) // EVERY
    return episodes


if __name__ == '__main__':
    import argparse
    ap = argparse.ArgumentParser()
    ap.add_argument('--levels', default='GoToRedBall,GoToLocal,PickupLoc,GoTo,BossLevel')
    ap.add_argument('--seeds', type=int, default=5)
    ap.add_argument('--steps', type=int, default=300)
    ap.add_argument('--policy', default='random')
    a = ap.parse_args()
    levels = list(orc.LEVELS) if a.levels == 'all' else a.levels.split(',')
    for lv in levels:
        ep = 0
        for s in range(a.seeds):
            ep += compare(lv, 100 + s, a.steps, a.policy, act_seed=s)
        print('%20s OK  (%d seeds x %d steps, %d episodes)' % (lv, a.seeds, a.steps, ep), flush=True)
