"""Pin the oracle's plant: C restatement vs golden vectors taken from the reference binaries (right-hand sides, logged
episodes, and the binaries' own outputs recorded by tests/golden/make_golden_refbin.py)."""
import os

import numpy as np
import pytest

from oracle import plant as P

G = os.path.join(os.path.dirname(__file__), 'golden')
KAT = np.load(os.path.join(G, 'plant_rhs_kat.npz'))
TRAJ = np.load(os.path.join(G, 'plant_traj_kat.npz'))
REFBIN = np.load(os.path.join(G, 'refbin_kat.npz'))


@pytest.mark.parametrize('variant', P.VARIANTS)
def test_port_rhs_bit_exact_vs_reference_binary_kat(variant):
    pl = P.PortPlant(variant)
    assert np.array_equal(pl.initial_state(), KAT[variant + '_ic'])
    X, U, F = KAT[variant + '_X'], KAT[variant + '_U'], KAT[variant + '_F']
    live = [i for i in range(19) if i not in (13, 14)]
    for x, u, f in zip(X, U, F):
        got = pl.rhs(x, u)
        assert np.array_equal(got[live], f[live])      # bit-exact, fp64


def _replay(pl, a):
    X = pl.initial_state()
    out, X = pl.step(X, np.zeros(10))            # reset(): one zero-command step (phlabenv.py:409-413)
    err = 0.0
    outs = []
    for k in range(a.shape[0]):
        cmd = np.zeros(10)
        cmd[:3] = a[k, 3:6]
        out, X = pl.step(X, cmd)
        outs.append(out)
        err = max(err, np.abs(out - a[k, 6:18]).max())
    return err, np.array(outs)


@pytest.mark.parametrize('key', sorted(TRAJ.files))
def test_port_replays_logged_reference_episodes(key):
    err, _ = _replay(P.PortPlant('h2000_v90'), TRAJ[key])
    assert err < 1e-12          # log files were written with np.savetxt (%.18e); survey measured <= 4.3e-14


@pytest.mark.parametrize('key', ['ERL10_rl_statehistory_episode209', 'l_TD3_rl_statehistory_episode575'])
def test_port_equals_reference_binary_on_episodes(key):
    e1, o1 = _replay(P.PortPlant('h2000_v90'), TRAJ[key])
    rows = REFBIN['replay_%s_rows' % key]
    assert rows[-1] == len(o1) - 1
    assert np.array_equal(o1[rows], REFBIN['replay_%s_out' % key])


@pytest.mark.parametrize('variant', ['ice', 'cg', 'h2000_v150'])
def test_port_equals_reference_binary_other_variants(variant):
    a = P.PortPlant(variant)
    Xa = a.initial_state()
    rng = np.random.RandomState(1)
    outs = []
    for k in range(300):
        cmd = np.zeros(10)
        cmd[:3] = 0.05 * rng.uniform(-1, 1, 3)
        oa, Xa = a.step(Xa, cmd)
        outs.append(oa)
    assert np.array_equal(np.array(outs)[REFBIN['seeded_%s_rows' % variant]], REFBIN['seeded_%s_out' % variant])
