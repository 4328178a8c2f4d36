"""Record what the reference's own plant binaries and Python modules return for the inputs of the tests that compare
against them, so that those tests run without the reference tree.  Needs the byte copies under oracle/_ref
(oracle/build.py) and the reference checkout's base/ directory:

    python tests/golden/make_golden_refbin.py <reference checkout>      -> tests/golden/refbin_kat.npz

Long trajectories are stored at a fixed subset of rows (every 20th step, every step around the switching times, the last
step) and long weight vectors at a fixed sample of coordinates (GENOME_SAMPLE), to keep the fixture small; the reference's
starting genomes, which the tests rebuild with oracle.actor.Actor, are pinned by a SHA-256 digest of their float32 bytes.
"""
import ctypes
import hashlib
import os
import shutil
import sys
import tempfile
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from oracle import build as obuild, fast, phlab, plant as P, refsig          # noqa: E402

D = ctypes.c_double
LIVE9 = [0, 1, 2, 3, 4, 5, 6, 7, 9]
GENOME_SAMPLE = 1024


def pulse_window(k):
    return 1996 <= k <= 2003 or 2296 <= k <= 2303 or k == 2150


def episode_rows(n):
    rows = set(range(0, n, 20)) | set(range(1990, 2010)) | set(range(2290, 2310)) | {n - 1}
    return np.array(sorted(r for r in rows if r < n), dtype=np.int32)


def gust_windows(out):
    """states of the gust / test binaries before and after the native calls around the 20-23 s pulse, stepped from
    initialize() with cmd = 0.02 sin(0.01 k + [0, 1, 2]) (tests/test_generated_plant.py, tests/test_boundary_gpu.py)."""
    for build in ('gust', 'test'):
        pl = P.RefPlant(build)
        X = pl.initial_state()
        ks, before, after = [], [], []
        for k in range(2306):
            cmd = 0.02 * np.sin(0.01 * k + np.arange(3))
            _, Xn = pl.step(X, np.concatenate([cmd, np.zeros(7)]))
            if pulse_window(k):
                ks.append(k); before.append(X); after.append(Xn)
            X = Xn
        out[build + '_k'] = np.array(ks, dtype=np.int32)
        out[build + '_X0'] = np.array(before)
        out[build + '_X1'] = np.array(after)


def lifter(out):
    """rt_GetLookupIndex / rt_Lookup / rt_Lookup2D_Normal of the h2000_v90 binary on the probes of
    tests/test_lifter_reference.py, in the order that test visits them."""
    sys.path.insert(0, os.path.join(ROOT, 'tests'))
    import test_lifter_reference as T
    fd, path = tempfile.mkstemp(suffix='.so'); os.close(fd)
    shutil.copy(os.path.join(obuild.HERE, '_ref', 'citation_h2000_v90.so'), path)
    L = ctypes.CDLL(path)
    L.rt_GetLookupIndex.restype = ctypes.c_int
    L.rt_GetLookupIndex.argtypes = [ctypes.POINTER(D), ctypes.c_int, D]
    L.rt_Lookup.restype = D
    L.rt_Lookup.argtypes = [ctypes.POINTER(D), ctypes.c_int, D, ctypes.POINTER(D)]
    L.rt_Lookup2D_Normal.restype = D
    L.rt_Lookup2D_Normal.argtypes = [ctypes.POINTER(D), ctypes.c_int, ctypes.POINTER(D), ctypes.c_int, ctypes.POINTER(D), D, D]
    idx = []
    rng = np.random.RandomState(0)
    for x in T.axes(rng):
        arr = (D * len(x))(*x)
        idx += [L.rt_GetLookupIndex(arr, len(x), float(u)) for u in T.probes(x, rng)]
    lk2, lk1 = [], []
    rng = np.random.RandomState(1)
    for _ in range(30):
        nx, ny = rng.randint(2, 12), rng.randint(2, 12)
        xs = np.sort(rng.uniform(-1, 1, nx)); ys = np.sort(rng.uniform(-1, 1, ny)); zs = rng.normal(0, 1, nx * ny)
        X, Y, Z = (D * nx)(*xs), (D * ny)(*ys), (D * (nx * ny))(*zs)
        for _ in range(20):
            x, y = rng.uniform(-1.3, 1.3), rng.uniform(-1.3, 1.3)
            lk2.append(L.rt_Lookup2D_Normal(X, nx, Y, ny, Z, x, y))
            lk1.append(L.rt_Lookup(X, nx, x, (D * nx)(*zs[:nx])))
    os.unlink(path)
    out['lookup_index'] = np.array(idx, dtype=np.int32)
    out['lookup2d'] = np.array(lk2)
    out['lookup1d'] = np.array(lk1)


def plant_replays(out):
    """outputs of the h2000_v90 binary replaying two logged episodes, and of three other builds under seeded commands
    (tests/test_oracle_plant.py)."""
    traj = np.load(os.path.join(HERE, 'plant_traj_kat.npz'))
    for key in ('ERL10_rl_statehistory_episode209', 'l_TD3_rl_statehistory_episode575'):
        pl = P.RefPlant('h2000_v90')
        a = traj[key]
        X = pl.initial_state()
        _, X = pl.step(X, np.zeros(10))
        outs = []
        for k in range(a.shape[0]):
            cmd = np.zeros(10)
            cmd[:3] = a[k, 3:6]
            o, X = pl.step(X, cmd)
            outs.append(o)
        rows = np.array(sorted(set(range(0, len(outs), 10)) | {len(outs) - 1}), dtype=np.int32)
        out['replay_%s_rows' % key] = rows
        out['replay_%s_out' % key] = np.array(outs)[rows]
    for variant in ('ice', 'cg', 'h2000_v150'):
        pl = P.RefPlant(variant)
        X = pl.initial_state()
        rng = np.random.RandomState(1)
        outs = []
        for k in range(300):
            cmd = np.zeros(10)
            cmd[:3] = 0.05 * rng.uniform(-1, 1, 3)
            o, X = pl.step(X, cmd)
            outs.append(o)
        rows = np.array(sorted(set(range(0, 300, 3)) | {299}), dtype=np.int32)
        out['seeded_%s_rows' % variant] = rows
        out['seeded_%s_out' % variant] = np.array(outs)[rows]


def closed_loop(out):
    """the oracle env on the cg_timed (40 s) and gust (30 s) binaries flown by the kernel-order SERL10 elite actor
    (tests/test_eval_suite_gpu.py): live states at episode_rows(), executed steps and return."""
    g = np.load(os.path.join(HERE, 'actors.npz'))['serl10_elite_h72_tanh']
    for name, mode, seed_base, t_max, smooth in (('cg_timed', 'cg-timed', 40, 40, 6.0), ('gust', 'gust', 41, 30, 4.5)):
        lv, st = refsig.make_ref_params(1, seed_base=seed_base, t_max=t_max)
        env = phlab.CitationEnv(mode, 'ref', t_max=t_max)
        env.smooth_w = smooth
        obs = env.reset(lv[0], st[0])
        tot, xs = 0.0, []
        for k in range(100 * t_max + 1):
            a = fast.actor_forward_kernel_order(g, np.asarray(obs, dtype=np.float32).reshape(1, 7), 72)[0]
            obs, rew, done, _ = env.step(a)
            xs.append(env.x.copy())
            tot += rew
            if done:
                break
        rows = episode_rows(len(xs))
        out[name + '_steps'] = np.int32(len(xs))
        out[name + '_return'] = np.float64(tot)
        out[name + '_rows'] = rows
        out[name + '_x'] = np.asarray(xs)[rows][:, LIVE9]


def genome_digest(G):
    return hashlib.sha256(np.ascontiguousarray(G, dtype=np.float32).tobytes()).hexdigest()


def reference_modules(out, ref):
    """base/core/mod_neuro_evo.py proximal_mutate and base/core/genetic_agent.py update_parameters on the seeded inputs of
    tests/test_evo_prox.py; the resulting genomes at GENOME_SAMPLE fixed coordinates."""
    cwd, work = os.getcwd(), tempfile.mkdtemp()
    os.chdir(work)                          # the reference's Parameters creates ./tmp/
    sys.path.insert(0, os.path.join(ref, 'base'))
    from core import mod_neuro_evo as ref_ne, genetic_agent as ref_ga
    from parameters import Parameters as RefP
    flat = lambda g: torch.cat([p.data.reshape(-1) for p in g.actor.parameters()])
    args = RefP(types.SimpleNamespace(pop_size=4, mut_type='proximal', env='x', frames=1, seed=1, disable_cuda=True))
    args.state_dim, args.action_dim, args.device = 7, 3, torch.device('cpu')
    torch.manual_seed(0)
    genes = [ref_ga.GeneticAgent(args) for _ in range(3)]
    G = torch.stack([flat(g) for g in genes])
    sample = np.sort(np.random.RandomState(0).choice(G.shape[1], GENOME_SAMPLE, replace=False)).astype(np.int32)
    states = torch.randn(3, 32, 7) * 0.1
    ssne = ref_ne.SSNE(args, None, None)

    class FakeBuf:
        def __init__(self, st):
            self.st = st

        def __len__(self):
            return 32

        def sample(self, n):
            return (self.st, None, None, None, None)
    for k, g in enumerate(genes):
        g.buffer = FakeBuf(states[k])
        torch.manual_seed(100 + k)
        ssne.proximal_mutate(g, mag=args.mutation_mag)
    out['genome_sample'] = sample
    out['proximal_G_init_sha256'] = np.array(genome_digest(G.numpy()))
    out['proximal_G_ref'] = torch.stack([flat(g) for g in genes])[:, sample].numpy()
    out['mutation_mag'] = np.float64(args.mutation_mag)

    torch.manual_seed(0)
    kids = [ref_ga.GeneticAgent(args) for _ in range(3)]
    p1s = [ref_ga.GeneticAgent(args) for _ in range(3)]
    p2s = [ref_ga.GeneticAgent(args) for _ in range(3)]
    out['distil_G_init_sha256'] = np.array(genome_digest(torch.stack([flat(g) for g in kids + p1s + p2s]).numpy()))
    lin = torch.nn.Linear(10, 2)

    def critic(s, a):
        q = lin(torch.cat((s, a), 1))
        return q[:, :1], q[:, 1:]
    states = torch.randn(3, 40, 7) * 0.2
    mse_ref = [kids[c].update_parameters((states[c], None, None, None, None), p1s[c].actor, p2s[c].actor, critic) for c in range(3)]
    out['distil_G_ref'] = torch.stack([flat(k) for k in kids])[:, sample].numpy()
    out['distil_mse_ref'] = np.asarray(mse_ref, dtype=np.float64)
    os.chdir(cwd)
    shutil.rmtree(work)


if __name__ == '__main__':
    assert obuild.have_ref() and os.path.exists(os.path.join(obuild.HERE, '_ref', 'citation_gust.so')), 'run oracle/build.py first'
    ref = os.path.abspath(sys.argv[1])
    out = {}
    gust_windows(out)
    lifter(out)
    plant_replays(out)
    closed_loop(out)
    reference_modules(out, ref)
    np.savez_compressed(os.path.join(HERE, 'refbin_kat.npz'), **out)
    print({k: v.shape for k, v in out.items()})
