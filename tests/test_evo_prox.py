"""N3: proximal / safe mutation batched over the population (serl_b200/evo_prox.py) against (a) the reference module itself
(base/core/mod_neuro_evo.py:183-252, results recorded in tests/golden/refbin_kat.npz) and (b) a per-actor autograd restatement."""
import hashlib
import os

import numpy as np
import torch

from oracle import actor as OA
from serl_b200 import evo, evo_prox

KAT = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'refbin_kat.npz'))


def per_actor_reference(genome, states, shape, activation, mag, delta):
    """the reference's algorithm on ONE actor with plain autograd over a functional forward."""
    G = genome.clone().reshape(1, -1).requires_grad_(True)
    out = evo_prox.actor_forward_batched(G, states[None], shape, activation)[0]
    mask = evo_prox.weight_mask(shape, G.device)
    jac = []
    for i in range(3):
        (g,) = torch.autograd.grad(out[:, i].sum(), G, retain_graph=True)
        jac.append(g[0, mask])
    scaling = torch.sqrt(sum(j ** 2 for j in jac))
    scaling[scaling == 0] = 1.0
    scaling[scaling < 0.01] = 0.01
    new = genome.clone()
    new[mask] = genome[mask] + delta / scaling
    return new


def test_batched_equals_per_actor_restatement():
    torch.manual_seed(3)
    shape = (7, 3, 32, 3)
    table, P = evo.param_table(*shape)
    G = torch.randn(6, P) * 0.2
    states = torch.randn(4, 20, 7) * 0.1
    idx = [5, 0, 3, 2]
    nw = int(evo_prox.weight_mask(shape, G.device).sum())
    delta = torch.randn(4, nw) * 0.02
    G2 = G.clone()
    evo_prox.proximal_mutate_batched(G2, idx, states, shape, 'tanh', 0.02, delta=delta)
    for k, i in enumerate(idx):
        want = per_actor_reference(G[i], states[k], shape, 'tanh', 0.02, delta[k])
        assert torch.allclose(G2[i], want, rtol=1e-5, atol=1e-6)
    assert torch.equal(G2[1], G[1]) and torch.equal(G2[4], G[4])          # untouched actors
    # biases / LayerNorm parameters are not mutated (extract_parameters takes 2-D parameters only, genetic_agent.py:125-135)
    m = evo_prox.weight_mask(shape, G.device)
    assert torch.equal(G2[:, ~m], G[:, ~m])


def reference_init(n):
    """n flat genomes drawn by the oracle's Actor (the reference's layer order and init draws) under the current torch seed."""
    return torch.from_numpy(np.stack([OA.flatten(OA.Actor()) for _ in range(n)]))


def check_reference_start(G, key):
    """the rebuilt starting genomes must be the reference's own: SHA-256 of their float32 bytes, recorded by
    tests/golden/make_golden_refbin.py."""
    digest = hashlib.sha256(np.ascontiguousarray(G.numpy(), dtype=np.float32).tobytes()).hexdigest()
    assert digest == str(KAT[key]), "the rebuilt starting genomes differ from the reference's: oracle.actor.Actor no longer draws like it"


def test_batched_proximal_mutation_equals_the_reference_module():
    """reference: SSNE.proximal_mutate (base/core/mod_neuro_evo.py:183-252) on three seeded actors, recorded at fixed
    genome coordinates by tests/golden/make_golden_refbin.py."""
    import torch.distributions as dist
    torch.manual_seed(0)
    G = reference_init(3)
    check_reference_start(G, 'proximal_G_init_sha256')
    shape = (7, 3, 72, 3)
    states = torch.randn(3, 32, 7) * 0.1
    mag = float(KAT['mutation_mag'])
    tot = int(evo_prox.weight_mask(shape, G.device).sum())          # Actor.count_parameters(): the 2-D weights
    deltas = []
    for k in range(3):
        torch.manual_seed(100 + k)
        deltas.append(dist.Normal(torch.zeros(tot), torch.ones(tot) * mag).sample())
    G2 = G.clone()
    evo_prox.proximal_mutate_batched(G2, [0, 1, 2], states, shape, 'tanh', mag, delta=torch.stack(deltas))
    cols = torch.as_tensor(KAT['genome_sample'], dtype=torch.long)
    G_ref = torch.as_tensor(KAT['proximal_G_ref'])
    assert (G_ref - G[:, cols]).abs().max() > 0.1
    assert (G2[:, cols] - G_ref).abs().max().item() <= 1e-6


def test_batched_distillation_step_equals_the_reference_update_parameters():
    """one Q-filtered behaviour-cloning Adam step (base/core/genetic_agent.py:22-60) for three children at once; reference
    genomes and losses recorded by tests/golden/make_golden_refbin.py."""
    from serl_b200 import evo_distil
    torch.manual_seed(0)
    G0, G1, G2 = reference_init(3), reference_init(3), reference_init(3)
    check_reference_start(torch.cat([G0, G1, G2]), 'distil_G_init_sha256')
    lin = torch.nn.Linear(10, 2)

    def critic(s, a):
        q = lin(torch.cat((s, a), 1))
        return q[:, :1], q[:, 1:]
    states = torch.randn(3, 40, 7) * 0.2
    shape = (7, 3, 72, 3)
    child = G0.clone().requires_grad_(True)
    opt = torch.optim.Adam([child], lr=1e-3)
    with torch.no_grad():
        a1 = evo_prox.actor_forward_batched(G1, states, shape, 'tanh')
        a2 = evo_prox.actor_forward_batched(G2, states, shape, 'tanh')
        fl = states.reshape(120, 7)
        q1 = torch.min(*critic(fl, a1.reshape(120, 3))).reshape(3, 40)
        q2 = torch.min(*critic(fl, a2.reshape(120, 3))).reshape(3, 40)
    opt.zero_grad()
    loss, mse = evo_distil.cloning_loss(evo_prox.actor_forward_batched(child, states, shape, 'tanh'), a1, a2, q1, q2)
    loss.backward()
    opt.step()
    cols = torch.as_tensor(KAT['genome_sample'], dtype=torch.long)
    G_ref = torch.as_tensor(KAT['distil_G_ref'])
    assert (G_ref - G0[:, cols]).abs().max() > 1e-4
    assert (child.detach()[:, cols] - G_ref).abs().max().item() <= 2e-6
    assert np.allclose(mse.numpy(), KAT['distil_mse_ref'], rtol=1e-4)


def test_sort_groups_by_fitness_order():
    from serl_b200 import evo_distil
    fit = {3: -10.0, 5: -2.0, 9: -7.0}
    g = evo_distil.sort_groups_by_fitness([3, 5, 9], fit)
    assert g[0][:2] == (5, 9) and g[-1][:2] == (9, 3) and g[0][2] == -9.0
