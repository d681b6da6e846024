"""RGB partial observations (RGBImgPartialObsWrapper, scripts/train_rl.py:54-58, babyai/evaluate.py:91-92): the pool's 513
pre-rendered tiles (csrc/rgb_tiles.h, a C++ rasteriser) against the oracle shim's literal restatement of gym_minigrid's
rendering code (oracle/shim/gym_minigrid/rendering.py + Grid.render_tile), whole images against the wrapper run on the
reference's own levels, and -- on the GPU -- the render kernel against both."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

ROOT = os.path.normpath(os.path.join(os.path.dirname(os.path.abspath(__file__)), '..'))
GOLD = os.path.join(ROOT, 'tests', 'golden', 'rgb_obs.npz')


def pool_tiles():
    from babyai_b200 import lib
    L = lib.load()
    t = np.zeros((513, 8, 8, 3), np.uint8)
    assert L.bb_rgb_tiles(t.ctypes.data_as(C.c_void_p)) == 0          # host-side rasteriser: no GPU involved
    return t


def assemble(obs, tiles):
    """numpy statement of what k_render_rgb does: obs uint8[n, 7, 7, 3] -> uint8[n, 56, 56, 3]"""
    obs = obs.reshape(-1, 7, 7, 3).astype(np.int64)
    cell = obs[..., 0] | (obs[..., 1] << 3) | (obs[..., 2] << 6)
    ids = np.where(obs[..., 0] == 0, 256, cell)
    ids[:, 3, 6] = np.where(obs[:, 3, 6, 0] == 0, 256, 257 + cell[:, 3, 6])
    img = tiles[ids]                                                   # [n, vi, vj, ty, tx, 3]
    return img.transpose(0, 2, 3, 1, 4, 5).reshape(-1, 56, 56, 3)      # pixel row = vj * 8 + ty, column = vi * 8 + tx


def shim_tile(cell_byte, agent, highlight):
    sys.path.insert(0, os.path.join(ROOT, 'oracle', 'shim'))
    from gym_minigrid.minigrid import Grid, _decode_obj
    t, c, s = cell_byte & 7, (cell_byte >> 3) & 7, cell_byte >> 6
    obj = _decode_obj(t, c, s) if t >= 2 else None
    return Grid.render_tile(obj, agent_dir=3 if agent else None, highlight=highlight, tile_size=8).astype(np.uint8)


def test_tiles_equal_shim_rasteriser():
    tiles = pool_tiles()
    n = 0
    for t in (1, 2, 4, 5, 6, 7):
        for c in range(6):
            for s in range(3):
                if t != 4 and s:
                    continue
                b = t | (c << 3) | (s << 6)
                assert np.array_equal(tiles[b], shim_tile(b, False, True)), (t, c, s)
                assert np.array_equal(tiles[257 + b], shim_tile(b, True, True)), ('agent', t, c, s)
                n += 1
    assert np.array_equal(tiles[256], shim_tile(0, False, False))
    assert n == 48


def test_golden_images_equal_tile_assembly():
    """tests/golden/rgb_obs.npz: (7x7x3 observation, 56x56x3 image) pairs produced by RGBImgPartialObsWrapper on the
    reference's levels (make_rgb_golden.py, build container)"""
    g = np.load(GOLD)
    assert np.array_equal(assemble(g['obs'], pool_tiles()), g['rgb'])


def test_wrapper_on_reference_levels_equals_tile_assembly():
    """observations of the reference's own levels under random actions (BossLevel, GoToLocal, Unlock; recorded in
    tests/golden/ref_rgb_levels.npz by make_ref_golden.py) through the shim's RGBImgPartialObsWrapper"""
    sys.path.insert(0, os.path.join(ROOT, 'oracle', 'shim'))
    from gym import spaces
    from gym_minigrid.minigrid import MiniGridEnv
    from gym_minigrid.wrappers import RGBImgPartialObsWrapper

    class View(MiniGridEnv):
        """what the wrapper reads of the env it wraps: the observation space and the view size"""
        def __init__(self):
            self.agent_view_size = 7
            self.observation_space = spaces.Dict({'image': spaces.Box(low=0, high=255, shape=(7, 7, 3), dtype='uint8')})
            self.action_space, self.reward_range, self.metadata = spaces.Discrete(7), (0, 1), {}
    w = RGBImgPartialObsWrapper(View())
    assert w.observation_space.spaces['image'].shape == (56, 56, 3)
    tiles = pool_tiles()
    z = np.load(os.path.join(ROOT, 'tests', 'golden', 'ref_rgb_levels.npz'))
    assert sorted(z.files) == ['BossLevel', 'GoToLocal', 'Unlock']
    for level in z.files:
        for t, raw in enumerate(z[level]):
            pic = w.observation({'image': raw, 'mission': ''})['image']
            assert np.array_equal(assemble(raw, tiles)[0], pic), (level, t)


@pytest.mark.gpu
def test_gpu_render_equals_tile_assembly_and_golden():
    import torch
    from babyai_b200 import BabyAIVecEnv
    tiles = pool_tiles()
    g = np.load(GOLD)
    env = BabyAIVecEnv('BossLevel', 333, seeds=np.arange(333, dtype=np.uint64) + 5)
    out = env.render_rgb(torch.as_tensor(g['obs']).cuda())
    assert np.array_equal(out.cpu().numpy(), g['rgb'])
    env.reset()
    acts = torch.randint(0, 7, (30, 333), device='cuda', dtype=torch.int8)
    for t in range(30):
        o, _r, _d = env.step(acts[t])
        assert np.array_equal(env.render_rgb().cpu().numpy(), assemble(o.cpu().numpy(), tiles)), t
    # a whole rollout buffer [T, N, 7, 7, 3] in one call
    T = 8
    obs = torch.zeros((T, 333, 7, 7, 3), dtype=torch.uint8, device='cuda')
    rew, done = torch.zeros((T, 333), device='cuda'), torch.zeros((T, 333), dtype=torch.uint8, device='cuda')
    env.rollout(acts[:T], obs, rew, done)
    pics = env.render_rgb(obs)
    assert pics.shape == (T, 333, 56, 56, 3)
    assert np.array_equal(pics.cpu().numpy().reshape(-1, 56, 56, 3), assemble(obs.cpu().numpy(), tiles))


@pytest.mark.gpu
def test_gpu_pixel_facades():
    """make_envs(pixel=True) / RGBImgPartialObsWrapper(envs): ParallelEnv returns {'image': uint8[56,56,3], 'mission'} dicts,
    DeviceParallelEnv keeps the pictures on the device."""
    from babyai_b200 import DeviceParallelEnv, ParallelEnv, RGBImgPartialObsWrapper, make_envs
    tiles = pool_tiles()
    envs = RGBImgPartialObsWrapper(make_envs('GoToLocal', 64))
    assert envs[0].observation_space.spaces['image'].shape == (56, 56, 3)
    pe, plain = ParallelEnv(envs), ParallelEnv(make_envs('GoToLocal', 64))
    o, p = pe.reset(), plain.reset()
    rng = np.random.RandomState(1)
    for t in range(20):
        assert all(np.array_equal(o[i]['image'], assemble(p[i]['image'], tiles)[0]) and o[i]['mission'] == p[i]['mission']
                   and 'direction' not in o[i] for i in range(64)), t
        a = rng.randint(0, 7, 64)
        o, r1, d1, _ = pe.step(a)
        p, r2, d2, _ = plain.step(a)
        assert r1 == r2 and d1 == d2
    de = DeviceParallelEnv(make_envs('GoToLocal', 64, pixel=True))
    b = de.reset()
    assert tuple(b.image.shape) == (64, 56, 56, 3) and b.image.is_cuda
    b, _r, _d, _i = de.step(rng.randint(0, 7, 64))
    assert tuple(b.image.shape) == (64, 56, 56, 3)
