"""The reference-facing surface on the GPU: batched plant C-ABI, CitationEnv per-step API, Agent.evaluate / train."""
import ctypes
import os
import random
import types

import numpy as np
import pytest
import torch

from oracle import actor as OA, phlab, plant as OP

pytestmark = pytest.mark.gpu


def make_args(folder, pop=6, hidden=16, **kw):
    from serl_b200.parameters import Parameters
    cla = types.SimpleNamespace(env='PHlab_attitude_nominal', seed=7, pop_size=pop, mut_type='normal', test_ea=True, **kw)
    os.makedirs(folder, exist_ok=True)
    cwd = os.getcwd(); os.chdir(folder)
    try:
        args = Parameters(cla)
    finally:
        os.chdir(cwd)
    args.save_foldername = str(folder) + '/'
    args.state_dim, args.action_dim, args.hidden_size = 7, 3, hidden
    return args


@pytest.mark.parametrize('variant', ['h2000_v90', 'ice', 'cg'])
def test_plant_step_kernel_matches_oracle(variant):
    from serl_b200 import _native, rollout
    L = _native.lib()
    dev = torch.device('cuda:0')
    n = 5
    v = torch.full((n,), rollout.PLANT_VARIANTS.index(variant), dtype=torch.int32, device=dev)
    X = torch.empty((n, 19), dtype=torch.float64, device=dev)
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    _native.check(L.serl_plant_init(ctypes.c_void_p(X.data_ptr()), ctypes.c_void_p(v.data_ptr()), n, st), 'init')
    pl = OP.PortPlant(variant)
    assert np.array_equal(X.cpu().numpy()[0], pl.initial_state())
    rng = np.random.RandomState(0)
    Xo = [pl.initial_state() for _ in range(n)]
    live = [0, 1, 2, 3, 4, 5, 6, 7, 9, 12, 15, 16, 17, 18]
    for k in range(200):
        cmd = 0.08 * rng.uniform(-1, 1, (n, 3))
        d = torch.as_tensor(cmd, device=dev)
        _native.check(L.serl_plant_step(ctypes.c_void_p(X.data_ptr()), ctypes.c_void_p(d.data_ptr()), ctypes.c_void_p(v.data_ptr()), n, st), 'step')
        for i in range(n):
            _, Xo[i] = pl.step(Xo[i], np.concatenate([cmd[i], np.zeros(7)]))
    got = X.cpu().numpy()
    ref = np.array(Xo)
    # same operation order in fp64; only libm (sin/cos/pow/exp: CUDA vs glibc, <= 2 ulp) differs
    assert np.abs(got[:, live] - ref[:, live]).max() < 1e-9
    assert np.allclose(got[:, live], ref[:, live], rtol=1e-11, atol=1e-12)


@pytest.mark.parametrize('build', ['gust', 'test'])
def test_timed_plant_step_api_flies_the_gust_pulse_like_the_binary(build):
    """serl_plant_step_timed with SERL_MODE_GUST (the per-step path of CitationEnv in 'gust' mode): one-step predictions from
    the binary's own states through both edges of the pulse (native calls 1996..2003, 2296..2303) and in its middle.  The
    binary's states before and after those calls are recorded in tests/golden/refbin_kat.npz (envs/test: the same pulse with
    the opposite sign)."""
    from serl_b200 import _native, rollout
    L = _native.lib()
    dev = torch.device('cuda:0')
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    kat = np.load(os.path.join(os.path.dirname(__file__), 'golden', 'refbin_kat.npz'))
    var = torch.tensor([rollout.mode_code(build) & ~0xff00], dtype=torch.int32, device=dev)
    live = [0, 1, 2, 3, 4, 5, 6, 7, 9, 12, 15, 16, 17, 18]
    worst, changed = 0.0, 0
    window = [k for k in range(2306) if 1996 <= k <= 2003 or 2296 <= k <= 2303 or k == 2150]
    assert kat[build + '_k'].tolist() == window
    for k, X0, X in zip(window, kat[build + '_X0'], kat[build + '_X1']):
        cmd = 0.02 * np.sin(0.01 * k + np.arange(3))
        Xd = torch.as_tensor(X0[None].copy(), device=dev)
        d = torch.as_tensor(cmd[None].copy(), device=dev)
        call = torch.tensor([k], dtype=torch.int32, device=dev)
        _native.check(L.serl_plant_step_timed(ctypes.c_void_p(Xd.data_ptr()), ctypes.c_void_p(d.data_ptr()), ctypes.c_void_p(var.data_ptr()),
                                              ctypes.c_void_p(call.data_ptr()), 1, st), 'serl_plant_step_timed')
        call0 = torch.tensor([0], dtype=torch.int32, device=dev)
        Xn = torch.as_tensor(X0[None].copy(), device=dev)
        _native.check(L.serl_plant_step_timed(ctypes.c_void_p(Xn.data_ptr()), ctypes.c_void_p(d.data_ptr()), ctypes.c_void_p(var.data_ptr()),
                                              ctypes.c_void_p(call0.data_ptr()), 1, st), 'serl_plant_step_timed')
        got = Xd.cpu().numpy()[0]
        worst = max(worst, np.abs(got[live] - X[live]).max())
        changed += int(np.abs(Xn.cpu().numpy()[0][live] - X[live]).max() > 1e-6)        # the same step outside the pulse (call 0)
    assert worst < 1e-9, worst
    assert changed >= 10


def test_citation_env_step_api_matches_oracle_env():
    from serl_b200.envs import config
    env = config.select_env('PHlab_attitude_nominal')
    np.random.seed(5)
    obs = env.reset()
    o_env = phlab.CitationEnv('nominal', 'auto')
    o_obs = o_env.reset(env.levels, env.starts)
    assert np.allclose(obs, o_obs)
    act = OA.unflatten(np.load(os.path.join(os.path.dirname(__file__), 'golden', 'actors.npz'))['serl10_elite_h72_tanh'], hidden=72)
    for k in range(150):
        a = act.select_action(o_obs)
        obs, r, d, info = env.step(a)
        o_obs, o_r, o_d, o_info = o_env.step(a)
        assert d == o_d and abs(r - o_r) < 1e-9 and np.abs(obs - o_obs).max() < 1e-9
    assert abs(info['t'] - o_info['t']) < 1e-12


def test_agent_evaluate_returns_reference_shaped_episode(tmp_path):
    from serl_b200.core import agent as agent_mod
    from serl_b200.envs import config
    args = make_args(tmp_path, pop=4, hidden=72)
    env = config.select_env('PHlab_attitude_nominal')
    torch.manual_seed(7); np.random.seed(7); random.seed(7)
    ag = agent_mod.Agent(args, env)
    w = np.load(os.path.join(os.path.dirname(__file__), 'golden', 'actors.npz'))['serl10_pop_h72_tanh']
    ag.pop.genomes.copy_(torch.as_tensor(w[:4]))
    np.random.seed(11)
    ag.gen_frames = 0
    ep = ag.evaluate(ag.pop[1], is_action_noise=False, store_transition=False)
    np.random.seed(11)
    levels, starts = env.draw_reference()
    o = phlab.run_episode(phlab.CitationEnv('nominal', 'auto'), OA.unflatten(w[1], hidden=72), levels, starts, record=True)
    assert len(ep.reward_lst) == o['steps'] == len(ep.state_history)
    assert abs(ep.fitness - o['fitness']) <= 1e-4 * abs(o['fitness'])
    assert abs(ep.length - o['t']) < 1e-12
    assert ep.actions.shape == (o['steps'], 3)
    assert ep.get_history().shape == (o['steps'], 19)
    # exploration episode stores transitions and keeps the np.random stream where the reference would leave it
    np.random.seed(3)
    ep2 = ag.evaluate(ag.rl_agent, is_action_noise=True, store_transition=True)
    n = len(ep2.reward_lst)
    after = np.random.rand()
    np.random.seed(3); env.draw_reference(); np.random.randn(n, 3)
    assert after == np.random.rand()
    assert len(ag.replay_buffer) == n and ag.num_frames == n


def test_agent_train_generations_and_checkpoint_format(tmp_path):
    from serl_b200.core import agent as agent_mod
    from serl_b200.envs import config
    args = make_args(tmp_path, pop=6, hidden=16)
    env = config.select_env('PHlab_attitude_nominal')
    torch.manual_seed(7); np.random.seed(7); random.seed(7)
    ag = agent_mod.Agent(args, env)
    before = ag.pop.genomes.clone()
    keys = {'best_train_fitness', 'test_score', 'test_sd', 'pop_avg', 'pop_min', 'elite_index', 'avg_smoothness', 'smoothness_sd',
            'rl_reward', 'rl_smoothness', 'rl_smoothness_std', 'rl_std', 'avg_ep_len', 'ep_len_sd', 'PG_obj', 'TD_loss', 'pop_novelty'}
    for gen in range(2):
        stats = ag.train()
        assert set(stats.keys()) == keys          # agent.py:297-315
        assert np.isfinite(stats['best_train_fitness']) and stats['pop_min'] <= stats['pop_avg'] <= stats['best_train_fitness']
        assert 0 <= stats['elite_index'] < 6
    assert not torch.equal(before, ag.pop.genomes)
    assert ag.num_frames > 0 and ag.num_episodes > 0
    assert set(ag.evolver.selection_stats) == {'elite', 'selected', 'discarded', 'total'} and ag.evolver.selection_stats['total'] >= 1
    ag.save_agent(args, stats['elite_index'])
    pop_dict = torch.load(os.path.join(args.save_foldername, 'evo_nets.pkl'), weights_only=False)
    assert sorted(pop_dict) == ['actor_%d' % i for i in range(6)]
    assert list(pop_dict['actor_0'])[:2] == ['net.0.weight', 'net.0.bias']
    oracle_actor = OA.from_state_dict(torch.load(os.path.join(args.save_foldername, 'elite_net.pkl'), weights_only=False), 'tanh')   # loads into the reference layout
    assert np.array_equal(OA.flatten(oracle_actor), ag.pop.genomes[int(stats['elite_index'])].cpu().numpy())


def _train_generations(folder, prefetch, n, poke=None):
    from serl_b200.core import agent as agent_mod
    from serl_b200.envs import config
    args = make_args(folder, pop=6, hidden=16)
    args.prefetch_generation = prefetch
    env = config.select_env('PHlab_attitude_nominal')
    torch.manual_seed(7); np.random.seed(7); random.seed(7)
    env.seed(7)
    ag = agent_mod.Agent(args, env)
    out, flags = [], []
    for g in range(n):
        if poke is not None and g == poke:
            ag.pop.genomes[2].mul_(0.5)          # the caller edits an actor between two generations
        out.append(ag.train())
        flags.append(ag.timing['front_prefetched'])
    torch.cuda.synchronize()
    return out, flags, ag


def test_next_generation_front_launched_ahead_changes_no_result(tmp_path):
    """train() queues the next generation's rollouts before waiting for its own validation scores; the statistics of
    every generation, the populations and the counters must equal those of strictly one generation per call."""
    a, fa, aga = _train_generations(tmp_path / 'a', True, 3)
    b, fb, agb = _train_generations(tmp_path / 'b', False, 3)
    assert fa == [0.0, 1.0, 1.0] and fb == [0.0, 0.0, 0.0]
    for x, y in zip(a, b):
        for k in x:
            assert (x[k] == y[k]) or (np.isnan(x[k]) and np.isnan(y[k])), k
    assert torch.equal(aga.pop.genomes, agb.pop.genomes)
    assert (aga.num_frames, aga.num_episodes) == (agb.num_frames, agb.num_episodes)
    assert len(aga.replay_buffer) == len(agb.replay_buffer)


def test_front_launched_ahead_is_dropped_when_the_population_changed(tmp_path):
    a, fa, _ = _train_generations(tmp_path, True, 3, poke=1)
    assert fa == [0.0, 0.0, 1.0]
    assert all(np.isfinite(s['best_train_fitness']) for s in a)


def test_smoothness_kernel_matches_reference_formula():
    """K6 vs calc_smoothness (base/core/utils.py:82-120) on real action histories, incl. an early-terminated episode."""
    from serl_b200 import rollout
    from serl_b200.core.utils import calc_smoothness
    from oracle import refsig
    acts = np.load(os.path.join(os.path.dirname(__file__), 'golden', 'actors.npz'))
    torch.manual_seed(7)
    w = np.concatenate([acts['serl10_pop_h72_tanh'][:2], np.stack([OA.flatten(OA.Actor(hidden=72)) for _ in range(2)])])
    lv, st = refsig.make_ref_params(3, seed_base=17)
    dev = torch.device('cuda:0')
    md = torch.tensor([rollout.mode_code(m) for m in ('nominal', 'be', 'ice')], dtype=torch.int32, device=dev)
    r = rollout.population_rollout(torch.as_tensor(w, device=dev), rollout.actor_shape(72), torch.as_tensor(lv, device=dev),
                                   torch.as_tensor(st, device=dev), md, actions=True)
    sm = rollout.smoothness(r.actions, r.steps).cpu().numpy()
    steps = r.steps.cpu().numpy()
    a = r.actions.cpu().numpy().astype(np.float64)
    assert (steps < 2001).any() and (steps == 2001).any()
    for i in range(4):
        for e in range(3):
            ref = calc_smoothness(a[i, e, :steps[i, e]])
            assert abs(sm[i, e] - ref) <= 2e-5 * abs(ref) + 1e-9, (i, e, sm[i, e], ref)


def test_evaluation_mode_80s_episode_matches_oracle():
    """set_eval_mode (envs/phlabenv.py:295-301): t_max = 80 s -> 8001 steps, reference widths scaled (block 16 s, smooth 13 s)."""
    from serl_b200 import rollout
    from oracle import refsig
    w = np.load(os.path.join(os.path.dirname(__file__), 'golden', 'actors.npz'))['serl10_elite_h72_tanh'][None]
    lv, st = refsig.make_ref_params(1, seed_base=80, t_max=80)
    assert 15.5 < st[0, 0, 1] < 16.5
    dev = torch.device('cuda:0')
    md = torch.tensor([rollout.mode_code('nominal')], dtype=torch.int32, device=dev)
    r = rollout.population_rollout(torch.as_tensor(w, device=dev), rollout.actor_shape(72), torch.as_tensor(lv, device=dev),
                                   torch.as_tensor(st, device=dev), md, horizon=8001, t_max=80.0, smooth_width=13.0)
    from test_rollout_gpu import _F64Actor
    env = phlab.CitationEnv('nominal', 'auto', t_max=80)
    act = OA.unflatten(w[0], hidden=72)
    o = phlab.run_episode(env, act, lv[0], st[0])
    o64 = phlab.run_episode(env, _F64Actor(act), lv[0], st[0])
    assert o['steps'] == 8001 and int(r.steps[0, 0]) == 8001
    # this 80 s flight bifurcates around t = 55 s: the oracle's own float32 vs float64 forward pass differ by 0.5 % in
    # return; same criterion as tests/test_rollout_gpu.py::check
    sens = abs(o64['fitness'] - o['fitness']) / abs(o['fitness'])
    assert abs(float(r.returns[0, 0]) - o['fitness']) <= max(1e-4, 4 * sens) * abs(o['fitness'])
    # and a well-conditioned prefix: the first 40 s (4001 steps) must agree tightly
    r40 = rollout.population_rollout(torch.as_tensor(w, device=dev), rollout.actor_shape(72), torch.as_tensor(lv, device=dev),
                                     torch.as_tensor(st, device=dev), md, horizon=4001, t_max=80.0, smooth_width=13.0)
    env40 = phlab.CitationEnv('nominal', 'auto', t_max=80)
    obs = env40.reset(lv[0], st[0]); tot = 0.0
    for _ in range(4001):
        obs, rew, done, _ = env40.step(act.select_action(obs)); tot += rew
    assert int(r40.steps[0, 0]) == 4001 and abs(float(r40.returns[0, 0]) - tot) <= 1e-4 * abs(tot)
