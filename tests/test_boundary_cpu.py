"""Host logic of the drop-in boundary that needs no GPU: genome views, checkpoint keys, sharding, fitness all-gather (gloo)."""
import os
import types

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

from oracle import actor as OA


def make_args(folder, pop=4, hidden=8):
    from serl_b200.parameters import Parameters
    cla = types.SimpleNamespace(env='PHlab_attitude_nominal', seed=7, pop_size=pop, mut_type='normal')
    cwd = os.getcwd(); os.chdir(folder)          # Parameters creates ./tmp/ for checkpoints
    try:
        args = Parameters(cla)
    finally:
        os.chdir(cwd)
    args.device = torch.device('cpu')
    args.state_dim, args.action_dim, args.hidden_size = 7, 3, hidden
    return args


def test_population_views_and_reference_init_order(tmp_path):
    from serl_b200.population import PopulationList
    args = make_args(tmp_path)
    torch.manual_seed(7)
    pop = PopulationList(args, device='cpu')
    torch.manual_seed(7)
    ref = [OA.Actor(hidden=8) for _ in range(4)]
    for a, r in zip(pop, ref):
        assert np.array_equal(a.actor.flat().numpy(), OA.flatten(r))        # same RNG consumption as Actor(args) x pop
    assert list(pop[0].actor.state_dict().keys())[:4] == ['net.0.weight', 'net.0.bias', 'net.2.weight', 'net.2.bias']
    assert 'net.3.gamma' in pop[0].actor.state_dict() and 'net.11.bias' in pop[0].actor.state_dict()
    # parameters are views of the genome matrix, both ways
    pop.genomes[2, 0] = 123.0
    assert pop[2].actor.net[0].weight.data[0, 0].item() == 123.0
    pop[1].actor.net[11].bias.data[2] = -5.0
    assert pop.genomes[1, -1].item() == -5.0
    obs = np.zeros(7)
    assert pop[0].actor.select_action(obs).shape == (3,)


def test_ssne_rejects_out_of_scope_operators(tmp_path):
    from serl_b200.core.mod_neuro_evo import SSNE
    args = make_args(tmp_path)
    args.mut_type = 'proximal'
    assert SSNE(args, None, None).mutate == 'proximal'        # batched on the device (serl_b200/evo_prox.py)
    args.distil_crossover, args.distil_type = True, 'fitness'
    assert SSNE(args, None, None).distil                      # batched on the device (serl_b200/evo_distil.py)
    args.distil_type = 'distance'
    with pytest.raises(NotImplementedError):
        SSNE(args, None, None)
    args.distil_crossover = False
    args.mut_type = 'bogus'
    with pytest.raises(ValueError):
        SSNE(args, None, None)


def test_select_env_names():
    from serl_b200.envs import config
    e = config.select_env('PHlab_attitude_nominal')
    assert e.action_space.shape[0] == 3 and e.observation_space.shape[0] == 7
    assert config.select_env('phlab_attitude_ice').variant == 'ice'
    assert config.select_env('phlab_attitude_be').fault == 'be'
    with pytest.raises(ValueError):
        config.select_env('phlab_attitude_bogus')
    with pytest.raises(ValueError):
        config.select_env('cartpole')


def test_shard_bounds_cover_population():
    from serl_b200 import engine
    for pop in (1, 7, 10, 512, 513):
        for world in (1, 2, 3, 8):
            b = [engine.shard_bounds(pop, world, r) for r in range(world)]
            assert b[0][0] == 0 and b[-1][1] == pop
            assert all(b[i][1] == b[i + 1][0] for i in range(world - 1))


def _worker(rank, world, port, pop, out):
    import torch.distributed as dist
    from serl_b200 import engine
    dist.init_process_group('gloo', init_method='tcp://127.0.0.1:%d' % port, rank=rank, world_size=world)
    full = torch.arange(pop, dtype=torch.float64) * 1.5 - 3.0
    lo, hi = engine.shard_bounds(pop, world, rank)
    got = engine.gather_fitness(full[lo:hi].clone(), pop, world, rank)
    out[rank] = bool(torch.equal(got, full))
    dist.destroy_process_group()


@pytest.mark.parametrize('pop', [7, 10])
def test_fitness_all_gather_world2_gloo(pop):
    mgr = mp.Manager()
    out = mgr.dict()
    port = 29500 + (os.getpid() + pop) % 2000
    mp.spawn(_worker, args=(2, port, pop, out), nprocs=2, join=True)
    assert out[0] and out[1]


def test_dropin_aliases_resolve_reference_import_names():
    """base/train.py:6-12 imports `core.agent`, `parameters.Parameters`, `core.utils.load_config`, `envs.config`."""
    import subprocess, sys
    code = ("import sys; sys.path.insert(0, %r); import serl_b200.dropin as d; d.install();"
            "from core import agent; from parameters import Parameters; from core.utils import load_config, Episode;"
            "import envs, envs.config; from core import mod_neuro_evo, genetic_agent, td3, replay_memory, mod_utils;"
            "assert agent.Agent.__module__ == 'serl_b200.core.agent'; assert hasattr(envs.config, 'select_env');"
            "print('ok')") % os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    p = subprocess.run([sys.executable, '-c', code], capture_output=True, text=True, cwd='/tmp')
    assert p.returncode == 0 and p.stdout.strip().endswith('ok'), p.stderr


def test_host_and_oracle_reference_signal_generators_agree():
    from serl_b200 import refsig as P
    from oracle import refsig as O
    a, b = P.make_ref_params(7, seed_base=99), O.make_ref_params(7, seed_base=99)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    for t in (0.0, 3.99, 4.5, 7.2, 19.99, 20.0):
        assert P.ref_value_deg(a[0][3, 0], a[1][3, 0], t, 0.21) == O.ref_value_deg(b[0][3, 0], b[1][3, 0], t, 0.21)


def test_calc_smoothness_matches_reference_formula_literal():
    """core/utils.calc_smoothness vs a literal transcription of base/core/utils.py:82-120 (loop over channels, scipy-style fft)."""
    from serl_b200.core.utils import calc_smoothness
    rng = np.random.RandomState(0)
    for n in (2001, 780, 16, 5):
        y = np.cumsum(rng.normal(0, 0.01, (n, 3)), axis=0)
        N, A, dt = y.shape[0], y.shape[1], 0.01
        T = N * dt
        freq = np.linspace(dt, 1 / (2 * dt), N // 2 - 1)
        Syy = np.zeros((N // 2 - 1, A))
        for i in range(A):
            Y = np.fft.fft(y[:, i], N)
            Syy[:, i] = np.abs(Y[1:N // 2] * np.conjugate(Y[1:N // 2])) * dt
        ref = -np.sqrt(np.sum(np.einsum('ij,i -> j', Syy, freq) * 2 / N)) * 100 * (80 / T)
        assert np.isclose(calc_smoothness(y), ref, rtol=1e-12, atol=0)


def test_device_replay_rings_keep_reference_ring_semantics():
    """DeviceReplayMemory / PopulationBuffers / ActorBuffer against the reference's list-with-position ring
    (base/core/replay_memory.py:40-62): same content in the same chronological order, for pushes that wrap and pushes
    longer than the capacity.  (Host logic; tensors on the CPU.)"""
    from serl_b200.core.replay_memory import ActorBuffer, DeviceReplayMemory, PopulationBuffers
    torch.manual_seed(0)
    for cap in (5, 8):
        ref = []                                                 # the reference ring as a plain list
        pos = 0
        dev = DeviceReplayMemory(cap, 'cpu')
        pa, pb = PopulationBuffers(3, cap, 'cpu'), PopulationBuffers(3, cap, 'cpu')
        for n in (3, 4, 9, 1, 12, 2):
            rows = torch.randn(n, 20)
            for r in rows:                                       # replay_memory.py:53-62 push()
                if len(ref) < cap:
                    ref.append(None)
                ref[pos] = r[:19]
                pos = (pos + 1) % cap
            dev.add_rows(rows)
            ActorBuffer(pa, 1).add_rows(rows)
            pb.append(torch.tensor([1]), rows[None], torch.ones((1, n), dtype=torch.bool))
            chrono = torch.stack(ref[pos:] + ref[:pos]) if len(ref) == cap else torch.stack(ref)
            assert torch.equal(dev._chronological_rows(), chrono)
            assert torch.equal(pa.rows_of(1), chrono) and torch.equal(pb.rows_of(1), chrono)
            assert torch.equal(pa.data, pb.data) and torch.equal(pa.pos, pb.pos) and torch.equal(pa.count, pb.count)
            assert len(dev) == len(ActorBuffer(pa, 1)) == len(ref)
        assert len(ActorBuffer(pa, 0)) == 0 and pa.rows_of(2).shape == (0, 19)
