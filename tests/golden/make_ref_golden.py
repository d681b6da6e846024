"""Records what the reference's own code computes for the comparisons that check this project against it, so that the
suite can replay them without the reference:

  ref_runs.npz              every run of tests/common.py reference_runs() (compare_ref.record: actions + state digests)
  ref_place_agent_hang.npz  MiniBossLevel seed 698: the 56 levels before the one RoomGrid.place_agent hangs on, and that
                            level's grid and rooms (tests/test_oracle_vs_reference.py)
  ref_demos.npz             demos of the reference's one-env-at-a-time loop (make_agent_demos.generate_demos;
                            tests/test_demos.py)
  ref_rgb_levels.npz        observations of the reference's levels under random actions (tests/test_rgb.py)

Needs the reference tree (refenv.REFERENCE).

usage: python tests/golden/make_ref_golden.py [runs|hang|demos|rgb ...]"""
import json
import os
import signal
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.normpath(os.path.join(HERE, '..', '..'))
sys.path[:0] = [ROOT, os.path.join(ROOT, 'oracle'), os.path.join(ROOT, 'tests')]
import compare_ref  # noqa: E402
import refenv  # noqa: E402
from common import reference_runs  # noqa: E402


def runs():
    """all runs end to end: keys[i] played steps[i] actions and stored ceil(steps[i] / EVERY) digests"""
    out = {}
    for _group, level, kw in reference_runs():
        key = compare_ref.run_key(level, **kw)
        if key not in out:
            out[key] = compare_ref.record(level, **kw)
    np.savez_compressed(os.path.join(HERE, 'ref_runs.npz'), keys=np.array(json.dumps(list(out))),
                        steps=np.array([len(a) for a, _ in out.values()], np.int32),
                        actions=np.concatenate([a for a, _ in out.values()]), checks=np.concatenate([c for _, c in out.values()]))
    print('%d runs' % len(out))


def hang():
    env = refenv.make_env('MiniBossLevel', 698)
    obs, missions = [], []
    for k in range(56):
        ob = env.reset()
        obs.append(ob['image'])
        missions.append(ob['mission'])

    class Hung(Exception):
        pass

    def on_alarm(*a):
        raise Hung()
    signal.signal(signal.SIGALRM, on_alarm)
    signal.alarm(3)
    try:
        env.reset()
        raise AssertionError('the 57th level of MiniBossLevel seed 698 did not hang')
    except Hung:
        pass
    finally:
        signal.alarm(0)
    e = env.unwrapped
    rooms = [(i, j, e.get_room(i, j)) for j in range(e.num_rows) for i in range(e.num_cols)]
    np.savez_compressed(os.path.join(HERE, 'ref_place_agent_hang.npz'), obs=np.stack(obs), missions=np.array(json.dumps(missions)),
                        hung_grid=e.grid.encode(), room_ij=np.array([(i, j) for i, j, _ in rooms]),
                        room_top=np.array([r.top for _, _, r in rooms]), room_size=np.array([r.size for _, _, r in rooms]))


def demos():
    """the arguments of tests/test_demos.py"""
    from test_demos import DEMO_LEVELS, demo_actions
    out = {}
    for level in DEMO_LEVELS:
        acts, seeds = demo_actions()
        T, n = acts.shape
        missions, images, directions, actions = [], [], [], []
        for k in range(n):
            env = refenv.make_env(level, seeds[k], 'philox')
            obs = env.reset()
            mission, imgs, dirs, acs = obs['mission'], [], [], []
            done, reward, t = False, 0, 0
            while not done and t < T:
                a = int(acts[t, k])
                new_obs, reward, done, _ = env.step(a)
                acs.append(a); imgs.append(obs['image']); dirs.append(obs['direction'])
                obs = new_obs
                t += 1
            if done and reward > 0:
                missions.append(mission); images += imgs; directions += dirs; actions += acs
        out[level + '.missions'] = np.array(json.dumps(missions))
        out[level + '.images'] = np.stack(images)
        out[level + '.directions'] = np.array(directions, np.int8)
        out[level + '.actions'] = np.array(actions, np.int8)
    np.savez_compressed(os.path.join(HERE, 'ref_demos.npz'), **out)


def rgb():
    gym = refenv.setup('philox')
    rng = np.random.RandomState(0)
    out = {}
    for level in ('BossLevel', 'GoToLocal', 'Unlock'):
        env = gym.make('BabyAI-%s-v0' % level)
        env.seed(11)
        env.reset()
        obs = []
        for t in range(120):
            a = int(rng.choice(7, p=[0.15, 0.15, 0.3, 0.15, 0.1, 0.13, 0.02]))
            raw, _r, done, _ = env.step(a)
            obs.append(raw['image'])
            if done:
                env.reset()
        out[level] = np.stack(obs)
    np.savez_compressed(os.path.join(HERE, 'ref_rgb_levels.npz'), **out)


if __name__ == '__main__':
    parts = sys.argv[1:] or ['runs', 'hang', 'demos', 'rgb']
    for p in parts:
        {'runs': runs, 'hang': hang, 'demos': demos, 'rgb': rgb}[p]()
        print(p, 'done', flush=True)
