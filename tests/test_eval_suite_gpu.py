"""SURVEY.md 8(f) N4 — the evaluation suite on the device: 80 s episodes on user-defined references
(base/evaluate.py:169-180), the sensor-noise shim (envs/noise/citation.py:72-82), nMAE (base/core/utils.py:39-58)."""
import os

import numpy as np
import pytest
import torch

from oracle import actor as A, phlab, refsig

pytestmark = pytest.mark.gpu
ACT = np.load(os.path.join(os.path.dirname(__file__), 'golden', 'actors.npz'))
REFBIN = np.load(os.path.join(os.path.dirname(__file__), 'golden', 'refbin_kat.npz'))


class KOActor:
    """the kernel-order actor (bit-exact with the GPU) with the select_action interface of the oracle env loop"""

    def __init__(self, g, hidden=72):
        self.g, self.hidden = g, hidden

    def select_action(self, obs):
        from oracle import fast
        return fast.actor_forward_kernel_order(self.g, np.asarray(obs, dtype=np.float32).reshape(1, 7), self.hidden)[0]


def test_sensor_noise_shim_matches_the_oracle_with_the_same_draws():
    from serl_b200 import rollout
    dev = torch.device('cuda:0')
    g = ACT['serl10_elite_h72_tanh']
    lv, st = refsig.make_ref_params(2, seed_base=31)
    horizon = 400
    z = np.random.RandomState(4).randn(1, 2, horizon + 1, 7).astype(np.float32)
    md = torch.zeros(2, dtype=torch.int32, device=dev)
    r = rollout.population_rollout(torch.as_tensor(g[None], device=dev), rollout.actor_shape(72), torch.as_tensor(lv, device=dev),
                                   torch.as_tensor(st, device=dev), md, horizon=horizon, trace=True, sensor_noise=torch.as_tensor(z, device=dev))
    torch.cuda.synchronize()
    clean = rollout.population_rollout(torch.as_tensor(g[None], device=dev), rollout.actor_shape(72), torch.as_tensor(lv, device=dev),
                                       torch.as_tensor(st, device=dev), md, horizon=horizon)
    for e in range(2):
        env = phlab.CitationEnv('nominal', 'auto')
        env.noise_z = z[0, e].astype(np.float64)
        obs = env.reset(lv[e], st[e])
        tot = 0.0
        xs = []
        for k in range(horizon):
            obs, rew, done, info = env.step(KOActor(g).select_action(obs))
            xs.append(env.x.copy())
            tot += rew
            if done:
                break
        assert int(r.steps[0, e]) == k + 1
        assert abs(float(r.returns[0, e]) - tot) <= 1e-6 * abs(tot)
        assert np.abs(r.trace_x[0, e, :k + 1].cpu().numpy()[:, :8] - np.asarray(xs)[:, :8]).max() < 1e-9
        assert abs(float(r.returns[0, e]) - float(clean.returns[0, e])) > 1e-3          # the noise is really applied


def test_validate_agent_on_user_references_matches_the_reference_loop():
    """base/evaluate.py:59-150 restated on the oracle env vs serl_b200.evaluation.validate_agent (one traced launch)."""
    from serl_b200 import evaluation, rollout, signals
    from serl_b200.envs import config
    from serl_b200.core.utils import calc_nMAE, calc_smoothness
    g = ACT['serl10_elite_h72_tanh']
    t_max = 80
    times = np.linspace(0., t_max, 6)
    refs = [(signals.SmoothedStepSequence(times, [0, 12, 3, -4, -8, 2], smooth_width=t_max // 10),
             signals.SmoothedStepSequence(times, [2, -2, 2, 10, 2, -6], smooth_width=t_max // 10)),
            (signals.SmoothedStepSequence(times, [0, -6, 6, 9, -3, 0], smooth_width=t_max // 10),
             signals.SmoothedStepSequence(times, [0, 5, -5, 0, 10, 0], smooth_width=t_max // 10))]
    env = config.select_env('PHlab_attitude_ice')
    env.set_eval_mode(t_max)
    data, stats = evaluation.validate_agent(g, rollout.actor_shape(72), env, refs, num_trails=1)
    # the reference's loop on the oracle env
    nm, sm = [], []
    for th, ph in refs:
        oenv = phlab.CitationEnv('ice', 'auto', t_max=t_max)
        oenv.smooth_w = float(th.smooth_width)
        obs = oenv.reset(np.stack([th.levels, ph.levels]), np.stack([th.starts, ph.starts]))
        done, errs, us = False, [], []
        while not done:
            x_ctrl = oenv.x[[7, 6, 5]].copy()
            us.append(oenv.last_u.copy())
            ref_value = np.deg2rad(oenv.ref_deg())
            obs, rew, done, _ = oenv.step(KOActor(g).select_action(obs))
            errs.append(ref_value - x_ctrl)
        nm.append(calc_nMAE(np.asarray(errs)))
        sm.append(calc_smoothness(np.asarray(us)))
    assert data.shape[1] == 3 + 3 + 12 + 1 and data.shape[0] == len(errs)
    assert abs(stats.nmae - np.average(nm)) <= 1e-5 * abs(np.average(nm)), (stats, nm)
    assert abs(stats.sm - np.average(sm)) <= 1e-5 * abs(np.average(sm)), (stats, sm)


def test_calc_nmae_literal():
    from serl_b200.core.utils import calc_nMAE
    e = np.random.RandomState(1).randn(500, 3) * 0.02
    mae = np.mean(np.absolute(e), axis=0)
    rng = np.array([np.deg2rad(20), np.deg2rad(20), max(np.abs(np.average(e[:, -1])), 3.14159 / 180)])
    assert calc_nMAE(e) == pytest.approx(np.mean(mae / rng) * 100, rel=1e-14)


def test_noise_mode_and_time_triggered_modes_are_named():
    from serl_b200.envs import config
    assert config.select_env('PHlab_attitude_noise').sensor_noise
    assert config.select_env('PHlab_attitude_cg-shift').mode == 'cg-timed'
    gust = config.select_env('PHlab_attitude_gust')
    assert gust.sensor_noise and gust.mode == 'gust' and gust.mode_code & (1 << 24)
    test = config.select_env('PHlab_attitude_test')
    assert not test.sensor_noise and test.mode == 'test' and (test.mode_code >> 24) == 3
    with pytest.raises(ValueError):
        config.select_env('PHlab_attitude_nosuchmode')


def test_cg_timed_build_switches_at_20_s_like_the_reference_binary():
    """envs/cg_timed ('CG Aft after 20s', envs/phlabenv.py:159-163): nominal dynamics until the model clock reaches 20 s — in the
    LAST ode5 stage of native call 1999 — then three moment-arm parameters change.  40 s episodes (4001 steps) through the
    kernel vs the reference binary stepped by the oracle env (recorded by tests/golden/make_golden_refbin.py: live states every
    20th step and around the switch, executed steps, return); also the plain cg and nominal modes must differ from it."""
    from serl_b200 import rollout
    dev = torch.device('cuda:0')
    g = ACT['serl10_elite_h72_tanh']
    lv, st = refsig.make_ref_params(1, seed_base=40, t_max=40)
    md = lambda m: torch.tensor([rollout.mode_code(m)], dtype=torch.int32, device=dev)
    run = lambda m: rollout.population_rollout(torch.as_tensor(g[None], device=dev), rollout.actor_shape(72), torch.as_tensor(lv, device=dev),
                                               torch.as_tensor(st, device=dev), md(m), horizon=4001, trace=True, t_max=40.0, smooth_width=6.0)
    r = run('cg-timed')
    torch.cuda.synchronize()
    r.check()
    n, tot, rows = int(REFBIN['cg_timed_steps']), float(REFBIN['cg_timed_return']), REFBIN['cg_timed_rows']
    assert int(r.steps[0, 0]) == n == 4001
    tx = r.trace_x[0, 0, :n].cpu().numpy()
    live = [0, 1, 2, 3, 4, 5, 6, 7, 9]
    assert np.abs(tx[rows][:, live] - REFBIN['cg_timed_x']).max() < 1e-8
    assert abs(float(r.returns[0, 0]) - tot) <= 1e-8 * abs(tot)
    nominal = run('nominal')
    assert np.array_equal(nominal.trace_x[0, 0, :1999].cpu().numpy()[:, live], tx[:1999, live])        # identical before the trigger
    assert np.abs(nominal.trace_x[0, 0, 2100:2400].cpu().numpy()[:, live] - tx[2100:2400, live]).max() > 1e-5


def test_gust_build_flies_the_pulse_like_the_reference_binary():
    """envs/gust ('Vertical Gust of 15ft/s at 20s', envs/phlabenv.py:165-169): nominal dynamics, and for 20 s <= t <= 23 s the
    aerodynamic angle of attack is alpha - atan(w / V).  A 30 s episode (3001 steps, sensor noise off) through the kernel vs the
    reference binary stepped by the oracle env (recorded by tests/golden/make_golden_refbin.py: live states every 20th step and
    around both edges of the pulse, executed steps, return); the untraced launch (stage derivatives in tensor memory) must
    return the same bits as the traced one (local memory)."""
    from serl_b200 import rollout
    dev = torch.device('cuda:0')
    g = ACT['serl10_elite_h72_tanh']
    lv, st = refsig.make_ref_params(1, seed_base=41, t_max=30)
    md = lambda m: torch.tensor([rollout.mode_code(m)], dtype=torch.int32, device=dev)
    run = lambda m, trace: rollout.population_rollout(torch.as_tensor(g[None], device=dev), rollout.actor_shape(72), torch.as_tensor(lv, device=dev),
                                                      torch.as_tensor(st, device=dev), md(m), horizon=3001, trace=trace, t_max=30.0, smooth_width=4.5,
                                                      gust=m == 'gust')
    r = run('gust', True)
    torch.cuda.synchronize()
    r.check()
    n, tot, rows = int(REFBIN['gust_steps']), float(REFBIN['gust_return']), REFBIN['gust_rows']
    assert int(r.steps[0, 0]) == n
    tx = r.trace_x[0, 0, :n].cpu().numpy()
    live = [0, 1, 2, 3, 4, 5, 6, 7, 9]
    err = np.abs(tx[rows][:, live] - REFBIN['gust_x']).max(axis=1)
    assert err.max() < 1e-8, (int(rows[err.argmax()]), float(err.max()))
    assert abs(float(r.returns[0, 0]) - tot) <= 1e-8 * abs(tot)
    nominal = run('nominal', True)
    assert np.array_equal(nominal.trace_x[0, 0, :1999].cpu().numpy()[:, live], tx[:1999, live])        # identical before the gust
    assert np.abs(nominal.trace_x[0, 0, 2100:2300].cpu().numpy()[:, live] - tx[2100:2300, live]).max() > 1e-4
    fast = run('gust', False)
    assert torch.equal(fast.returns, r.returns) and torch.equal(fast.steps, r.steps)
    # a gust env in a launch made without the flag is reported, not silently flown as nominal
    bad = rollout.population_rollout(torch.as_tensor(g[None], device=dev), rollout.actor_shape(72), torch.as_tensor(lv, device=dev),
                                     torch.as_tensor(st, device=dev), md('gust'), horizon=50)
    with pytest.raises(Exception, match='gust'):
        bad.check()
