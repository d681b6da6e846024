"""GPU tests added after the last GPU visit of round 1 (the GPU budget was spent): they sort after
test_gpu_parity.py so that `-x` reaches them last.  Their logic is exercised in the GPU-less suite through the host
build of the kernel source (test_hostemu.py, test_learner_adapters.py); here the CUDA pool itself is on the other end."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from common import GOLDEN_LEVELS, GOLDEN_LEVELS_GPU, replay_golden  # noqa: E402
from test_gpu_parity import GpuPool  # noqa: E402


NEW_LEVELS = ['GoToImpUnlock', 'Unlock']          # generator kernel k_gen<true> / UNTR step kernels: never run on a GPU before


@pytest.mark.parametrize('level', [lv for lv in GOLDEN_LEVELS if lv not in GOLDEN_LEVELS_GPU and lv not in NEW_LEVELS])
def test_gpu_replays_remaining_golden(level):
    """Reference-generated traces (tests/golden/make_golden.py) of the served levels test_gpu_parity.py does not replay."""
    replay_golden(level, lambda lv, n, s: GpuPool(lv, n, s), lambda p, i: p.mission(i))


@pytest.mark.parametrize('level,n,fused_io', [('PutNextLocal', 96, False), ('GoToSeqS5R2', 64, False), ('BossLevel', 40, False),
                                               ('PutNextLocal', 96, True), ('BossLevel', 40, True)])
def test_device_parallel_env_and_preprocessor(level, n, fused_io):
    """babyai_b200.learner: observations stay in HBM between the step kernel and the learner's tensors."""
    import torch
    import oracle as orc
    from babyai_b200 import DeviceParallelEnv, ObssPreprocessor, make_envs
    from babyai_b200.levels import VOCAB
    T = 70
    env = DeviceParallelEnv(make_envs(level, n, seed=1), fused_io=fused_io)       # True: bb_pool_step_learner
    assert env.fused_io == fused_io
    o = orc.OraclePool(level, n, np.array([100 + i for i in range(n)], dtype=np.uint64))
    pre = ObssPreprocessor()
    obs = env.reset()
    assert obs.image.is_cuda and np.array_equal(obs.image.cpu().numpy(), o.reset())
    rng = np.random.RandomState(2)
    history, images, missions = [], [], []
    for t in range(T):
        p = pre(obs, device='cuda')
        assert p.image.is_cuda and p.image.dtype == torch.float32 and p.instr.dtype == torch.long
        ms = [o.mission(i) for i in range(n)]
        width = max(len(m.replace(',', '').split()) for m in ms)
        want = [[VOCAB.index(w) for w in m.replace(',', '').split()] for m in ms]
        assert p.instr.cpu().tolist() == [w + [0] * (width - len(w)) for w in want]
        assert obs[n - 1]['mission'] == ms[n - 1] and obs[0]['direction'] == int(o.direction[0])
        history.append(obs); images.append(p.image.clone()); missions.append(want)
        act = rng.randint(0, 7, n)
        obs, rew, done, info = env.step(act if t % 2 else torch.as_tensor(act, device='cuda'))
        oo, orr, od = o.step(act.astype(np.int8))
        assert np.array_equal(obs.image.cpu().numpy(), oo)
        assert np.array_equal(np.asarray(rew, dtype=np.float32).view(np.uint32), orr.view(np.uint32))
        assert np.array_equal(np.asarray(done), od.astype(bool))
    flat = [history[i][j] for j in range(n) for i in range(T)]          # rl/algos/base.py:208-210
    p = pre(flat, device='cuda')
    assert p.image.shape == (n * T, 7, 7, 3)
    want_img = torch.stack(images).transpose(0, 1).reshape(n * T, 7, 7, 3)
    assert torch.equal(p.image, want_img)
    width = p.instr.shape[1]
    rows = [missions[i][j] + [0] * (width - len(missions[i][j])) for j in range(n) for i in range(T)]
    assert p.instr.cpu().tolist() == rows
    assert env.pool.counters()['errors'] == 0


def test_own_arm_json_line():
    from test_bench_contract import BASE_KEYS, _line
    d = _line(['--steps', '80', '--warmup', '40', '--envs', '4096', '--no-cpu-baseline', '--no-other-configs'])
    assert (BASE_KEYS - {'cpu_baseline'}) | {'roofline', 'clocks', 'per_step_api', 'counters', 'learner_path'} <= set(d)
    r = d['roofline']
    assert r['bound'] == 'hbm' and r['unit'] == 'GB/s' and r['achieved'] > 0 and abs(r['frac'] - r['achieved'] / r['peak']) < 1e-9
    assert d['e2e']['h2d_bytes_per_step'] == 4096 and d['e2e']['d2h_bytes_per_step'] == 4096 * 153
    # the roofline comes from the SAME timed region as `value`, which covers exactly the requested steps
    assert d['steps'] == d['steps_requested'] == 80
    assert abs(d['value'] / d['n_gpus'] * 153 / 1e9 - r['achieved']) <= 1e-6 * r['achieved'] and r['kernel_frac'] > 0
    assert abs(d['ms_per_step'] * d['steps'] * 1e-3 * d['value'] - d['steps'] * 4096) <= 1e-3 * d['steps'] * 4096
    assert d['e2e']['steps'] >= 200 and d['per_step_api']['steps'] >= 200 and d['e2e']['per_rank']['min'] > 0
    assert d['reference_parallel_env']['available'] is False and d['facade_e2e']['value'] > 0
    assert d['gpu_launches'] > 0 and d['counters']['errors'] == 0 and d['dtype'] == 'u8'
    assert 'error' not in d['learner_path']['tensor_copies'] and 'error' not in d['learner_path']['fused_io'], d['learner_path']


def test_own_arm_dumps_the_last_timed_step(tmp_path):
    """--dump-outputs: the last of exactly --steps timed steps (here two whole rollouts of 40 and one of 10), the same on
    every run, and equal to the C oracle stepped through the warm-up and the timed steps with the same seeds and actions"""
    import torch
    import oracle as orc
    from test_bench_contract import _line
    from babyai_b200.sharding import shard_seeds
    n, T, warm, K = 4096, 40, 80, 90
    outs = []
    for k in range(2):
        d = _line(['--lean', '--steps', str(K), '--warmup', '40', '--envs', str(n), '--no-cpu-baseline', '--no-other-configs',
                   '--dump-outputs', str(tmp_path / str(k))])
        assert d['steps'] == K and d['warmup'] == warm
        outs.append({f: np.load(str(tmp_path / str(k) / (f + '.npy'))) for f in ('obs', 'reward', 'done', 'direction')})
    assert all(a.dtype == np.float32 for a in outs[0].values()) and outs[0]['obs'].shape == (n, 7, 7, 3)
    assert all(np.array_equal(outs[0][f], outs[1][f]) for f in outs[0])
    acts = torch.randint(0, 7, (T, n), device='cuda', dtype=torch.int8,
                         generator=torch.Generator(device='cuda').manual_seed(1234)).cpu().numpy()
    ref = orc.OraclePool('GoToLocal', n, shard_seeds(1, n, 0, 1))
    ref.reset()
    for t in list(range(T)) * ((warm + K) // T) + list(range((warm + K) % T)):
        o, r, dn = ref.step(acts[t], nthreads=16)
    assert np.array_equal(outs[0]['obs'], o.astype(np.float32)) and np.array_equal(outs[0]['reward'], r)
    assert np.array_equal(outs[0]['done'], dn.astype(np.float32))
    assert np.array_equal(outs[0]['direction'], np.asarray(ref.direction, np.float32))


# ---- from here on: kernels instantiated after the last GPU visit (k_gen<true>, k_step8<*, true>, k_rollout<1, true>) ----
@pytest.mark.parametrize('level', NEW_LEVELS)
def test_gpu_replays_new_level_golden(level):
    replay_golden(level, lambda lv, n, s: GpuPool(lv, n, s), lambda p, i: p.mission(i))


@pytest.mark.parametrize('level,n,steps,p', [('GoToImpUnlock', 256, 300, None),
                                              ('GoToImpUnlock', 128, 400, [0.12, 0.12, 0.30, 0.17, 0.14, 0.13, 0.02]),
                                              ('Unlock', 256, 300, None),
                                              ('Unlock', 128, 500, [0.12, 0.12, 0.30, 0.17, 0.14, 0.13, 0.02])])
def test_gpu_matches_oracle_new_levels(level, n, steps, p):
    """Levels added after the last GPU visit: k_gen (one warp per level) + k_step8 against the C oracle."""
    import oracle as orc
    from common import compare_pools
    seeds = np.array([100 + i for i in range(n)], dtype=np.uint64)
    g = GpuPool(level, n, seeds)
    compare_pools(orc.OraclePool(level, n, seeds), g, n, steps, act_seed=3, action_p=p, state=(n <= 128),
                  mission_a=lambda q, i: q.mission(i), mission_b=lambda q, i: q.mission(i))
    assert g.env.counters()['errors'] == 0


@pytest.mark.parametrize('level', ['GoToImpUnlock', 'Unlock'])
def test_rollout_equals_stepwise_new_levels(level):
    import torch
    from babyai_b200 import BabyAIVecEnv
    n, T = 300, 16
    seeds = np.arange(n, dtype=np.uint64) + 77
    a, b = BabyAIVecEnv(level, n, seeds=seeds), BabyAIVecEnv(level, n, seeds=seeds)
    acts = torch.randint(0, 7, (T, n), device='cuda', dtype=torch.int8)
    a.reset(); b.reset()
    obs = torch.zeros((T, n, 7, 7, 3), dtype=torch.uint8, device='cuda')
    rew = torch.zeros((T, n), device='cuda')
    done = torch.zeros((T, n), dtype=torch.uint8, device='cuda')
    for rep in range(2):
        a.rollout(acts, obs, rew, done)
        for t in range(T):
            o, r, d = b.step(acts[t])
            assert torch.equal(o, obs[t]) and torch.equal(r, rew[t]) and torch.equal(d, done[t]), (rep, t)
    assert a.counters()['errors'] == 0


@pytest.mark.parametrize('level,n,T', [('GoToLocal', 4096, 24), ('GoToLocal', 1000, 40), ('PickupLoc', 200, 40), ('GoToObjS4', 256, 40),
                                        ('PutNextLocal', 333, 32), ('BossLevel', 512, 16), ('GoToObjMazeS4R2', 300, 40), ('Unlock', 200, 16)])
def test_rollout_equals_stepwise(level, n, T):
    """bb_pool_rollout (persistent kernels: bulk tile stores, warp-cooperative swap-in, fused generator warp) == T x
    bb_pool_step (and, transitively, the oracle), directions and counters included; ragged sizes included."""
    import torch
    from babyai_b200 import BabyAIVecEnv
    seeds = np.arange(n, dtype=np.uint64) + 77
    a = BabyAIVecEnv(level, n, seeds=seeds)
    b = BabyAIVecEnv(level, n, seeds=seeds)
    acts = torch.randint(0, 7, (T, n), device='cuda', dtype=torch.int8)
    a.reset(); b.reset()
    obs = torch.zeros((T, n, 7, 7, 3), dtype=torch.uint8, device='cuda')
    rew = torch.zeros((T, n), device='cuda')
    done = torch.zeros((T, n), dtype=torch.uint8, device='cuda')
    dirs = torch.zeros((T, n), dtype=torch.int8, device='cuda')
    for rep in range(3):
        a.rollout(acts, obs, rew, done, dirs)
        for t in range(T):
            o, r, d = b.step(acts[t])
            assert torch.equal(o, obs[t]) and torch.equal(r, rew[t]) and torch.equal(d, done[t]) and torch.equal(b.direction, dirs[t]), (rep, t)
    assert a.counters() == b.counters() and a.counters()['errors'] == 0


@pytest.mark.timeout(600)
def test_c5_per_gpu_share_matches_oracle_slice():
    """BASELINE config 5 at its per-GPU size: BossLevel, 32 768 envs with the seeds rank 3 of 8 owns in the 262 144-env job
    (sharding.shard_seeds), 25 rollouts of 40 steps through k_rollout_cta with the generation passes running beside them
    (one pass overlaps several launches).  The first 512 envs are compared step by step with the C oracle on the same
    seeds and actions; a second pool with the same seeds must reproduce the last launch bit for bit (determinism under the
    asynchronous level supply); no ring may run dry."""
    import torch
    import oracle as orc
    from babyai_b200 import BabyAIVecEnv
    from babyai_b200.sharding import shard_seeds
    n, T, L, m = 32768, 40, 25, 512
    seeds = shard_seeds(1, 8 * n, 3, 8)
    assert seeds[0] == 100 + 3 * n
    pools = [BabyAIVecEnv('BossLevel', n, seeds=seeds) for _ in range(2)]
    ref = orc.OraclePool('BossLevel', m, seeds[:m])
    gen = torch.Generator(device='cuda').manual_seed(9)
    acts = torch.randint(0, 7, (L, T, n), device='cuda', dtype=torch.int8, generator=gen)
    bufs = [(torch.zeros((T, n, 7, 7, 3), dtype=torch.uint8, device='cuda'), torch.zeros((T, n), device='cuda'),
             torch.zeros((T, n), dtype=torch.uint8, device='cuda'), torch.zeros((T, n), dtype=torch.int8, device='cuda')) for _ in pools]
    o0 = pools[0].reset().cpu().numpy()
    pools[1].reset()
    assert np.array_equal(o0[:m], ref.reset())
    for k in range(L):
        pools[0].rollout(acts[k], *bufs[0])
        ho, hr, hd = bufs[0][0][:, :m].cpu().numpy(), bufs[0][1][:, :m].cpu().numpy(), bufs[0][2][:, :m].cpu().numpy()
        a = acts[k][:, :m].cpu().numpy()
        for t in range(T):
            oo, rr, dd = ref.step(a[t], nthreads=16)
            assert np.array_equal(ho[t], oo), (k, t)
            assert np.array_equal(hr[t].view(np.uint32), rr.view(np.uint32)) and np.array_equal(hd[t], dd), (k, t)
    for k in range(L):
        pools[1].rollout(acts[k], *bufs[1])
    torch.cuda.synchronize()
    assert all(bool(torch.equal(x, y)) for x, y in zip(bufs[0], bufs[1]))
    c0, c1 = pools[0].counters(), pools[1].counters()
    assert c0 == c1 and c0['errors'] == 0 and c0['steps'] == n * T * L and c0['episodes'] > 0


@pytest.mark.parametrize('level', ['GoToObjMazeS4R2', 'MiniBossLevel'])
def test_many_envs_facades_on_a_multi_room_level(level):
    """babyai.evaluate.ManyEnvs surface (evaluate.py:58-81) on the GPU for a multi-room level: vecenv.ManyEnvs (host dicts) and
    learner.DeviceManyEnvs (observations resident on the device) -- seed(seeds), reset(), step() that freezes finished envs
    and repeats their last result -- against the C oracle stepped without auto-reset, two evaluation chunks in a row."""
    import oracle as orc
    from babyai_b200 import DeviceManyEnvs, ManyEnvs, make_envs
    n = 48
    host, devm = ManyEnvs(make_envs(level, n)), DeviceManyEnvs(make_envs(level, n))
    rng = np.random.RandomState(4)
    for chunk in range(2):
        seeds = [10 ** 9 + chunk * n + k for k in range(n)]              # evaluate.py:105: seed + i * num_envs + k
        host.seed(seeds); devm.seed(seeds)
        ref = orc.OraclePool(level, n, np.array(seeds, dtype=np.uint64))
        oh, od, oo = host.reset(), devm.reset(), ref.reset()
        assert all(np.array_equal(oh[i]['image'], oo[i]) and oh[i]['mission'] == ref.mission(i) for i in range(n))
        assert np.array_equal(od.image.cpu().numpy(), oo)
        frozen, last = np.zeros(n, bool), [None] * n
        for t in range(160):
            act = rng.choice(7, size=n, p=[0.12, 0.12, 0.4, 0.1, 0.1, 0.14, 0.02])
            oh, rh, dh, _ = host.step(act)
            od, rd, dd, _ = devm.step(act)
            oo, ro, do = ref.step(act.astype(np.int8), autoreset=False)
            img = od.image.cpu().numpy()
            for i in range(n):
                want = last[i] if frozen[i] else (oo[i].copy(), float(ro[i]), bool(do[i]))
                assert np.array_equal(oh[i]['image'], want[0]) and np.array_equal(img[i], want[0]), (level, chunk, t, i)
                assert rh[i] == rd[i] == np.float32(want[1]) and dh[i] == dd[i] == want[2], (level, chunk, t, i)
                if not frozen[i] and do[i]:
                    frozen[i], last[i] = True, want
        assert host.pool.counters()['errors'] == 0 and devm.pool.counters()['errors'] == 0
