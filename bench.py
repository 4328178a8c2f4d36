#!/usr/bin/env python
"""Benchmark of the per-generation fitness hot path (BASELINE.json metric: env-steps/s).

    python bench.py --gpus N --steps K --warmup W            our arm (CUDA, one rank per GPU under torchrun)
    python bench.py --impl reference --gpus N --steps K ...  reference arm: the reference's CPU path (native plant
                                                             binary + batch-1 torch actor + numpy wrapper) on host cores

A "step" = one population evaluation (one generation's rollouts): pop x envs trajectories of up to 2001 plant steps.
Workload = BASELINE.json configs[2]: PH-LAB nominal h2000_v90, pop=512, 128 envs, 2001-step horizon, actor h=72 L=3 tanh.
The population is the shipped SERL10 checkpoint tiled to pop with N(0,1e-3) weight noise (trained actors fly the full
horizon; SURVEY.md 8(d) mode ii); executed steps are counted from the kernel's own step counters, not assumed.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

POP, N_ENVS, HORIZON, HIDDEN = 512, 128, 2001, 72
BYTES_PER_STEP = 208.0          # SURVEY.md 8(d): state round-trip model, the HBM denominator BASELINE.md asks for
FLOP_PER_STEP_F64 = 6 * 900.0   # generated RHS: ~700 fp64 flops + ~65 table interpolations per stage, 6 stages (DESIGN.md)
FLOP_PER_STEP_F32 = 34600.0     # actor h=72 L=3 (SURVEY.md 8(d))


def population(pop, seed=7):
    acts = np.load(os.path.join(ROOT, 'tests', 'golden', 'actors.npz'))
    base = acts['serl10_pop_h72_tanh']
    rng = np.random.RandomState(seed)
    w = base[np.arange(pop) % base.shape[0]].astype(np.float32)
    w = w + rng.normal(0, 1e-3, size=w.shape).astype(np.float32)
    return np.ascontiguousarray(w)


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get('hbm_gbs', 6650.0), 'measured'
    return 6650.0, 'fallback'


class ClockSampler:
    def __init__(self, idx):
        self.p = None
        self.path = '/tmp/serl_clocks_%d.csv' % os.getpid()
        try:
            self.p = subprocess.Popen(
                ['nvidia-smi', '-i', str(idx), '--query-gpu=clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,'
                 'clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
                 'clocks_event_reasons.sw_power_cap', '--format=csv,noheader,nounits', '-lms', '200'],
                stdout=open(self.path, 'w'), stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': []}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            pass
        sm, mx, reasons = [], [], set()
        for line in open(self.path):
            f = [x.strip() for x in line.split(',')]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), f[4:8]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        if sm:
            out = {'sm_mhz': float(np.median(sm)), 'sm_max_mhz': float(max(mx)), 'reasons': sorted(reasons), 'samples': len(sm)}
        return out


# ------------------------------------------------------------------------------------------------ reference arm
def _cpu_worker(args):
    import torch
    torch.set_num_threads(1)
    from oracle import actor as A, phlab
    w, jobs, lv, st = args
    env = phlab.CitationEnv('nominal', 'auto')
    steps = 0
    t0 = time.perf_counter()
    for a, e in jobs:
        act = A.unflatten(w[a], hidden=HIDDEN)
        steps += phlab.run_episode(env, act, lv[e], st[e])['steps']
    return steps, time.perf_counter() - t0


def host_cores():
    """usable host cores: os.cpu_count() capped by the cgroup CPU quota (the GPU boxes expose 128 CPUs but grant 16)."""
    n = os.cpu_count() or 1
    try:
        q, per = open('/sys/fs/cgroup/cpu.max').read().split()
        if q != 'max':
            n = max(1, min(n, int(int(q) / int(per))))
    except Exception:
        pass
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    return n


def cpu_reference_throughput(n_episodes_per_core=1, cores=None):
    """The reference's CPU execution model (one process per core, each with its own copy of the native plant binary,
    batch-1 torch forward, numpy wrapper) on a bounded sample of the bench workload."""
    import multiprocessing as mp
    from oracle import refsig, build as ob
    ob.build()
    cores = cores or host_cores()
    os.environ.setdefault('OMP_NUM_THREADS', '1')
    os.environ.setdefault('MKL_NUM_THREADS', '1')
    w = population(8)
    lv, st = refsig.make_ref_params(8)
    jobs = [[((c * n_episodes_per_core + i) % 8, (c + i) % 8) for i in range(n_episodes_per_core)] for c in range(cores)]
    ctx = mp.get_context('spawn')
    t0 = time.perf_counter()
    with ctx.Pool(cores) as pool:
        res = pool.map(_cpu_worker, [(w, j, lv, st) for j in jobs])
    wall = time.perf_counter() - t0
    steps = sum(r[0] for r in res)
    busy = max(r[1] for r in res)
    return steps / busy, steps, cores, wall, ('reference' if ob.have_ref() else 'port')


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    vals = []
    kind = 'port'
    for i in range(args.warmup + args.steps):
        v, steps, cores, wall, kind = cpu_reference_throughput(n_episodes_per_core=2)
        if i >= args.warmup:
            vals.append((v, steps, wall))
    v = float(np.mean([x[0] for x in vals]))
    sample = '%d cores x 2 episodes (<=2001 steps each) of the pop=512 x 128-env workload per step' % cores
    line = {
        'impl': 'reference', 'metric': 'env_steps_per_sec', 'value': v, 'unit': 'env-steps/s', 'n_gpus': args.gpus, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': 1e3 * float(np.mean([x[2] for x in vals])), 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
        'config': {'workload': 'PH-LAB nominal h2000_v90, pop=512, 128 envs, 2001-step horizon, actor h=72 L=3 tanh (bounded sample)'},
        'cpu_baseline': {'value': v, 'unit': 'env-steps/s', 'cores': cores, 'kind': kind, 'sample': sample},
        'e2e': {'value': v, 'unit': 'env-steps/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------ our arm
CFG4_MODES = ['nominal', 'be', 'jr', 'sa', 'se', 'ice', 'cg']        # BASELINE config 4: fault / plant mode randomised per env


def mixed_modes(n_envs, seed=7):
    rs = np.random.RandomState(seed)
    return [CFG4_MODES[i] for i in rs.randint(0, len(CFG4_MODES), n_envs)]


def timed_region(step_fn, steps, warmup, flush, sync_all):
    """W warm-up steps, then exactly K steps bracketed by barrier + synchronize; CUDA events on the launching stream.
    Returns (elapsed ms of the K steps, mean per-step kernel ms, last result)."""
    import torch
    res = None
    for _ in range(warmup):
        flush.zero_()
        res = step_fn(res)
    sync_all()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    t_begin, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    t_begin.record()
    for i in range(steps):
        flush.zero_()
        ev[i][0].record()
        res = step_fn(res)
        ev[i][1].record()
    t_end.record()
    sync_all()
    return t_begin.elapsed_time(t_end), float(np.mean([a.elapsed_time(b) for a, b in ev])), res


def agent_train_timing(dev, pop, n_envs, generations=6, prefetch=True):
    """Generations through the public API (Agent.train, base/core/agent.py:211-315 mirror) at the bench configuration,
    EA loop only (-test_ea: no TD3 gradient steps; the RL exploration + validation episodes still fly).  Median wall clock
    between successive returns of train(), no device synchronisation added between the calls (a training loop has none); with
    prefetch=False every call is followed by a full device synchronise (strictly one generation per call)."""
    import random
    import types
    import torch
    from serl_b200.core import agent as agent_mod
    from serl_b200.envs import config as env_config
    from serl_b200.parameters import Parameters
    cla = types.SimpleNamespace(env='PHlab_attitude_nominal', pop_size=pop, test_ea=True, num_envs=n_envs, seed=7, mut_type='normal',
                                should_log=False, frames=10 ** 9)
    cwd = os.getcwd()
    os.chdir('/tmp')
    try:
        args = Parameters(cla)
    finally:
        os.chdir(cwd)
    env = env_config.select_env(args.env_name)
    args.action_dim, args.state_dim = env.action_space.shape[0], env.observation_space.shape[0]
    torch.manual_seed(7); np.random.seed(7); random.seed(7)
    env.seed(7)
    args.prefetch_generation = bool(prefetch)
    ag = agent_mod.Agent(args, env)
    ag.pop.genomes.copy_(torch.from_numpy(population(pop)).to(dev))
    stamps, stats = [], None
    torch.cuda.synchronize()
    for g in range(generations + 1):
        stats = ag.train()
        if not prefetch:
            torch.cuda.synchronize()
        stamps.append(time.perf_counter())
    ag.last_timing = dict(ag.timing)
    torch.cuda.synchronize()                  # the front launched for a generation nobody asks for
    gaps = [1e3 * (b - a) for a, b in zip(stamps[:-1], stamps[1:])]
    ag.generation_gaps_ms = gaps
    return float(np.median(gaps)), stats, ag


def dump_outputs(out_dir, res, fit_all):
    """What the last timed step handed its caller: per-trajectory returns and executed steps of this rank's population
    [pop, n_envs] and the gathered per-actor fitness [pop_total], as float64 .npy files (1.05 MB at the bench size)."""
    os.makedirs(out_dir, exist_ok=True)
    for name, t in (('returns', res.returns), ('steps', res.steps), ('fitness', fit_all)):
        np.save(os.path.join(out_dir, name + '.npy'), t.detach().cpu().numpy().astype(np.float64))


def run_ours(args):
    import torch
    import torch.distributed as dist
    from serl_b200 import rollout, _native, engine
    from serl_b200 import refsig
    if not os.path.exists(_native.LIB_PATH):      # normally prebuilt in-tree; build the CUDA extension if it is not there
        if int(os.environ.get('LOCAL_RANK', '0')) == 0:
            from serl_b200 import build as _b
            _b.build()
        else:
            for _ in range(600):
                if os.path.exists(_native.LIB_PATH):
                    break
                time.sleep(0.5)

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise SystemExit('bench.py: no CUDA device (the product path has no CPU fallback)')
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    strong = args.scaling == 'strong'

    sh = rollout.actor_shape(HIDDEN, 3, 'tanh')
    lv_np, st_np = refsig.make_ref_params(N_ENVS)
    lv_host = torch.from_numpy(lv_np).pin_memory()
    st_host = torch.from_numpy(st_np).pin_memory()
    nominal = torch.full((N_ENVS,), rollout.mode_code('nominal'), dtype=torch.int32)
    mixed = torch.tensor([rollout.mode_code(m) for m in mixed_modes(N_ENVS)], dtype=torch.int32)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)      # > 126 MB L2

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def make_workload(pop_total_or_local, modes_host, shard):
        """device tensors of one workload: weak = `POP` actors per rank (rank-specific population), strong / config 4 = ONE
        population of POP actors, identical on every rank, each rank flies its contiguous shard."""
        if shard:
            w_all = population(POP, seed=7)
            lo, hi = engine.shard_bounds(POP, world, rank)
            w_host = torch.from_numpy(np.ascontiguousarray(w_all[lo:hi])).pin_memory()
        else:
            w_host = torch.from_numpy(population(POP, seed=7 + rank)).pin_memory()
        md_host = modes_host.pin_memory()
        return {'w_host': w_host, 'md_host': md_host, 'w': w_host.to(dev), 'lv': lv_host.to(dev), 'st': st_host.to(dev),
                'md': md_host.to(dev), 'order': rollout.variant_sorted_order(md_host.to(dev)), 'pop_total': POP if shard else POP * world}

    def make_step(wl):
        fit_all = wl['fit_all'] = torch.empty((wl['pop_total'],), dtype=torch.float64, device=dev)

        def one_step(res=None):
            r = rollout.population_rollout(wl['w'], sh, wl['lv'], wl['st'], wl['md'], horizon=HORIZON, out=res, env_order=wl['order'])
            fit_all.copy_(engine.gather_fitness(r.fitness, wl['pop_total'], world, rank))     # THE collective of the path
            return r
        return one_step

    def measure(wl, steps, warmup):
        elapsed_ms, kern_ms, res = timed_region(make_step(wl), steps, warmup, flush, sync_all)
        local_steps = int(res.steps.sum().item())
        res.check()
        stats = torch.tensor([elapsed_ms, kern_ms], dtype=torch.float64, device=dev)
        tot = torch.tensor([float(local_steps)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(stats, op=dist.ReduceOp.MAX)
            dist.all_reduce(tot, op=dist.ReduceOp.SUM)
        elapsed_ms, kern_ms = stats.tolist()
        return {'elapsed_ms': elapsed_ms, 'kern_ms': kern_ms, 'total_steps': tot.item(), 'value': tot.item() * steps / (elapsed_ms * 1e-3),
                'res': res}

    # ---- headline: weak scaling = BASELINE config 3 per GPU; strong = BASELINE config 4 (one pop = 512, mixed faults) sharded
    wl = make_workload(POP, mixed if strong else nominal, shard=strong)
    launches0 = _native.lib().serl_launch_count()
    sampler = ClockSampler(local) if rank == 0 else None
    m = measure(wl, args.steps, args.warmup)
    clocks = sampler.stop() if sampler else None
    launches = (_native.lib().serl_launch_count() - launches0) // (args.steps + args.warmup) * args.steps
    res = m['res']
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, res, wl['fit_all'])

    # ---- end to end through the public API with host buffers (H2D genomes + env params, D2H fitness) every step
    pop_local = wl['w'].shape[0]
    fit_host = torch.empty((wl['pop_total'],), dtype=torch.float64).pin_memory()
    h2d = wl['w_host'].numel() * 4 + lv_host.numel() * 8 + st_host.numel() * 8 + wl['md_host'].numel() * 4
    d2h = fit_host.numel() * 8

    def e2e_step(res):
        # the call a user makes: host genomes + env parameters in, fitness out; H2D of this rank's inputs and D2H of the
        # gathered fitness are inside the timed region
        wl['w'].copy_(wl['w_host'], non_blocking=True)
        wl['lv'].copy_(lv_host, non_blocking=True)
        wl['st'].copy_(st_host, non_blocking=True)
        wl['md'].copy_(wl['md_host'], non_blocking=True)
        r = rollout.population_rollout(wl['w'], sh, wl['lv'], wl['st'], wl['md'], horizon=HORIZON, out=res, env_order=wl['order'])
        fit_host.copy_(engine.gather_fitness(r.fitness, wl['pop_total'], world, rank), non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return r

    res = e2e_step(res)
    sync_all()
    t0 = torch.cuda.Event(enable_timing=True); t1 = torch.cuda.Event(enable_timing=True)
    t0.record()
    n_e2e = max(1, min(args.steps, 3))
    for _ in range(n_e2e):
        res = e2e_step(res)
    t1.record()
    sync_all()
    e2e_ms = torch.tensor([t0.elapsed_time(t1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_ms, op=dist.ReduceOp.MAX)
    e2e_value = m['total_steps'] * n_e2e / (e2e_ms.item() * 1e-3)

    # ---- the other scaling mode as a second, shorter measurement (same barrier / max-over-ranks timing)
    other = None
    if not args.no_generation:
        wl2 = make_workload(POP, nominal if strong else mixed, shard=not strong)
        m2 = measure(wl2, 2, 1)
        other = {'scaling': 'weak' if strong else 'strong',
                 'workload': ('BASELINE config 3 per GPU (pop=512/GPU, nominal)' if strong else
                              'BASELINE config 4: ONE population of 512 actors sharded over the GPUs, fault/plant mode per env uniform over '
                              '{nominal,be,jr,sa,se,ice,cg}, identical population on every rank'),
                 'value': m2['value'], 'unit': 'env-steps/s', 'ms_per_step': m2['elapsed_ms'] / 2, 'executed_steps_per_step': m2['total_steps'],
                 'note': 'strong scaling is bounded by the serial latency of one 2001-step trajectory (about 0.11 s for a warp alone on an '
                         'SM): with 64 actors x 4 warps per GPU the SMs hold 2 resident warps instead of 8'}
        del wl2, m2

    # ---- one full generation (rollout + SSNE.epoch: K2 select, host RNG planner, K3-K5), rank-local, and Agent.train()
    gen_ms = epoch_timing = smooth_timing = extras = agent_line = None
    if world == 1 and not args.no_generation:
        import random
        from serl_b200 import evo
        np.random.seed(7); random.seed(7)
        w = wl['w'].clone()
        times = []
        for _ in range(2):
            g0 = torch.cuda.Event(enable_timing=True); g1 = torch.cuda.Event(enable_timing=True)
            g0.record()
            r = rollout.population_rollout(w, sh, wl['lv'], wl['st'], wl['md'], horizon=HORIZON, out=res)
            _, plan = evo.epoch_flat(w, r.fitness, (7, 3, HIDDEN, 3))
            epoch_timing = plan.timing
            g1.record(); torch.cuda.synchronize()
            times.append(g0.elapsed_time(g1))
        gen_ms = float(np.mean(times))
        # the action-smoothness metric of every episode (K6; agent.py:128-134, -smooth_fitness)
        s0 = torch.cuda.Event(enable_timing=True); s1 = torch.cuda.Event(enable_timing=True); s2 = torch.cuda.Event(enable_timing=True)
        s0.record()
        r = rollout.population_rollout(wl['w'], sh, wl['lv'], wl['st'], wl['md'], horizon=HORIZON, actions=True)
        s1.record()
        sm = rollout.smoothness(r.actions, r.steps)
        s2.record(); torch.cuda.synchronize()
        smooth_timing = {'rollout_with_action_history_ms': s0.elapsed_time(s1), 'smoothness_kernel_ms': s1.elapsed_time(s2),
                         'action_history_bytes': int(r.actions.numel() * 4)}
        del r, sm, w

        def timed_rollout(genomes, modes_t, n_envs=N_ENVS, lvx=None, stx=None):
            a0 = torch.cuda.Event(enable_timing=True); a1 = torch.cuda.Event(enable_timing=True)
            lvx = wl['lv'] if lvx is None else lvx
            stx = wl['st'] if stx is None else stx
            rollout.population_rollout(genomes, sh, lvx, stx, modes_t, horizon=HORIZON)       # warm
            a0.record()
            rr = rollout.population_rollout(genomes, sh, lvx, stx, modes_t, horizon=HORIZON)
            a1.record(); torch.cuda.synchronize()
            n = int(rr.steps.sum().item())
            return {'executed_env_steps': n, 'ms': a0.elapsed_time(a1), 'env_steps_per_sec': n / (a0.elapsed_time(a1) * 1e-3),
                    'mean_episode_steps': n / float(rr.steps.numel())}
        # (i) reference-termination mode (SURVEY 8(d)): generation-0 (random-init) actors crash early; only executed steps count
        import types
        from serl_b200.core import genetic_agent
        torch.manual_seed(7)
        a_ns = types.SimpleNamespace(hidden_size=HIDDEN, num_layers=3, activation_actor='tanh', state_dim=7, action_dim=3)
        w0 = torch.stack([genetic_agent.Actor(a_ns).flat() for _ in range(POP)]).to(dev)
        extras = {'random_init_population': timed_rollout(w0, wl['md'])}
        # (ii) BASELINE config 2: pop = 50 (SERL50), 64 envs
        lv2, st2 = refsig.make_ref_params(64)
        extras['config2_pop50_64envs'] = timed_rollout(torch.from_numpy(population(50)).to(dev), wl['md'][:64].contiguous(), 64,
                                                       torch.as_tensor(lv2, device=dev), torch.as_tensor(st2, device=dev))
        # (iii) per-GPU share of config 4 on 8 GPUs: 64 actors x 128 envs
        extras['pop64_128envs'] = timed_rollout(wl['w'][:64].contiguous(), wl['md'])
        # ---- the public API: Agent.train() generations at the bench configuration
        if not args.no_agent:
            ag_ms, ag_stats, ag = agent_train_timing(dev, POP, N_ENVS)
            strict_ms, strict_stats, ag1 = agent_train_timing(dev, POP, N_ENVS, generations=3, prefetch=False)
            agent_line = {'generation_ms': ag_ms, 'population_rollout_ms': m['kern_ms'], 'ratio_to_population_rollout': ag_ms / m['kern_ms'],
                          'what': 'median wall clock between successive returns of Agent.train() (EA loop, -test_ea): RL exploration, RL validation and '
                                  'champion validation episodes (5 x 2001-step trajectories, ~0.11 s of serial latency each) fly on side streams '
                                  'and spare SMs; train() queues the next generation\'s rollouts before it waits for its own validation scores, '
                                  'so the validation latency overlaps the next population rollout',
                          'frames_per_generation': int(ag.gen_frames), 'test_score': float(ag_stats['test_score']),
                          'generation_gaps_ms': ag.generation_gaps_ms, 'phases_ms_last_generation': ag.last_timing,
                          'one_generation_per_call': {'generation_ms': strict_ms, 'ratio_to_population_rollout': strict_ms / m['kern_ms'],
                                                      'what': 'prefetch_generation=False, device synchronised after every call; speculative '
                                                              'validation of the previous elites instead',
                                                      'phases_ms_last_generation': ag1.last_timing,
                                                      'speculative_champion_validation': {'hits': int(ag1.spec_hits), 'tries': int(ag1.spec_tries)}}}
            del ag, ag1

    if rank == 0:
        peak, how = peaks()
        traffic = None
        for name in ('r02_rollout_traffic.json', 'r01_rollout_traffic.json'):
            tpath = os.path.join(ROOT, 'profiles', name)
            if os.path.exists(tpath):
                traffic = json.load(open(tpath)).get('dram_bytes_per_launch')
                break
        per_gpu_steps = m['total_steps'] / world
        kern_ms = m['kern_ms']
        achieved = BYTES_PER_STEP * per_gpu_steps / (kern_ms * 1e-3) / 1e9
        workload = ('BASELINE config 4: PH-LAB mixed faults per env, ONE pop=512 sharded over %d GPU(s), 128 envs, 2001-step horizon, h=72 L=3 tanh'
                    % world if strong else
                    'BASELINE config 3: PH-LAB nominal h2000_v90, pop=512/GPU, 128 envs, 2001-step horizon, actor h=72 L=3 tanh')
        line = {
            'metric': 'env_steps_per_sec', 'value': m['value'], 'unit': 'env-steps/s', 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
            'ms_per_step': m['elapsed_ms'] / args.steps, 'higher_is_better': True, 'scaling': args.scaling, 'vs_baseline': None,
            'dtype': 'f64 plant + f32 actor', 'data': 'synthetic',
            'config': {'workload': workload + '; SERL10 checkpoint tiled + N(0,1e-3) noise; executed steps counted by the kernel',
                       'pop_per_gpu': pop_local, 'pop_total': wl['pop_total'], 'n_envs': N_ENVS, 'horizon': HORIZON, 'hidden': HIDDEN,
                       'executed_steps_per_step': m['total_steps'], 'l2': 'flushed between timed iterations (256 MiB memset)',
                       'parallelism': 'population sharded over %d GPU(s), one NCCL all-gather of fitness per step' % world},
            'clocks': clocks,
            'e2e': {'value': e2e_value, 'unit': 'env-steps/s', 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h},
            'gpu_launches': int(launches),
            'gpu_launches_per_step': 'genome_layout (K0) + rollout_kernel_persist (K1) + fitness_mean',
            'other_scaling_mode': other,
            'generation_ms': gen_ms, 'epoch_breakdown': (epoch_timing if gen_ms is not None else None), 'agent_train': agent_line,
            'smoothness': smooth_timing, 'other_workloads': extras,
            'roofline': {'bound': 'hbm', 'achieved': achieved, 'peak': peak, 'unit': 'GB/s', 'frac': achieved / peak, 'traffic': traffic,
                         'peak_source': how, 'kernel': 'rollout_kernel_persist', 'kernel_ms': kern_ms,
                         'note': 'BASELINE metric denominator (208 B/env-step state round-trip model); the kernel keeps state on chip and is '
                                 'bound by fp64/fp32 issue, see fp_issue',
                         'fp_issue': {'f64_gflops': FLOP_PER_STEP_F64 * per_gpu_steps / (kern_ms * 1e-3) / 1e9,
                                      'f32_gflops': FLOP_PER_STEP_F32 * per_gpu_steps / (kern_ms * 1e-3) / 1e9}},
        }
        if world == 1 and not args.no_cpu:
            v, steps, cores, wall, kind = cpu_reference_throughput(n_episodes_per_core=3)
            # a tougher CPU number next to the reference's own execution model: the same path as optimised C + OpenMP
            # (oracle/fast.py; plant restatement + fp32 forward + wrapper, no Python / torch per-step dispatch)
            from oracle import fast
            from serl_b200 import refsig as _rs
            cw = population(2 * cores)
            clv, cst = _rs.make_ref_params(8)
            t0 = time.perf_counter()
            _, cstp = fast.evaluate_population(cw, HIDDEN, clv, cst, ['nominal'] * 8, threads=cores)
            c_port = {'value': float(cstp.sum() / (time.perf_counter() - t0)), 'unit': 'env-steps/s', 'cores': cores, 'kind': 'port',
                      'sample': '%d actors x 8 envs (%d env-steps), C + OpenMP whole-episode port' % (2 * cores, int(cstp.sum()))}
            line['cpu_baseline'] = {'value': v, 'unit': 'env-steps/s', 'cores': cores, 'kind': kind, 'optimised_c_port': c_port,
                                    'sample': '%d cores x 3 episodes (%d env-steps total, ~20 s of CPU work) of the same workload, one process per core' % (cores, steps)}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    # exactly ONE line on stdout (the JSON): libraries that print there (NCCL's version banner) are sent to stderr
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(real_stdout, 'w')
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=3)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--no-cpu', action='store_true', help='skip the cpu_baseline leg')
    ap.add_argument('--no-generation', action='store_true', help='skip the rollout+epoch generation timing and the other-workload legs')
    ap.add_argument('--no-agent', action='store_true', help='skip the Agent.train() timing')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write the returns, executed steps and gathered fitness of the last timed step to DIR/<name>.npy (CUDA arm only)')
    ap.add_argument('--scaling', default='weak', choices=['weak', 'strong'],
                    help='weak: BASELINE config 3 per GPU (pop=512/GPU); strong: BASELINE config 4 (ONE pop=512, mixed faults, sharded)')
    args = ap.parse_args()
    if args.impl == 'reference' and args.dump_outputs:
        ap.error('--dump-outputs writes what the CUDA path computed; the reference arm only measures throughput')
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_ours(args)


if __name__ == '__main__':
    main()
