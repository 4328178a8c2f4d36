"""Drop-in boundary (SURVEY.md 8(b)): the copy-free launcher examples/train.py drives the call sequence of the reference's
base/train.py (:54-139) through the same classes and must leave the three checkpoint files with the reference's key names."""
import os
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ARGS = ['-frames', '6000', '-pop_size', '6', '-mut_type', 'normal', '-test_ea']


def check_checkpoints(folder):
    pop = torch.load(os.path.join(folder, 'evo_nets.pkl'), weights_only=False)
    assert sorted(pop) == ['actor_%d' % i for i in range(6)]
    keys = ['net.0.weight', 'net.0.bias', 'net.2.weight', 'net.2.bias', 'net.3.gamma', 'net.3.beta', 'net.5.weight', 'net.5.bias',
            'net.6.gamma', 'net.6.beta', 'net.8.weight', 'net.8.bias', 'net.9.gamma', 'net.9.beta', 'net.11.weight', 'net.11.bias']
    assert list(pop['actor_0']) == keys                                   # base/core/genetic_agent.py:78-101 module tree
    assert list(torch.load(os.path.join(folder, 'elite_net.pkl'), weights_only=False)) == keys
    assert list(torch.load(os.path.join(folder, 'rl_net.pkl'), weights_only=False)) == keys


@pytest.mark.gpu
def test_copy_free_launcher_runs_the_train_py_call_sequence(tmp_path):
    p = subprocess.run([sys.executable, os.path.join(ROOT, 'examples', 'train.py')] + ARGS, cwd=tmp_path, capture_output=True, text=True,
                       timeout=1800)
    assert p.returncode == 0, p.stderr[-3000:]
    assert 'Frames:' in p.stdout
    check_checkpoints(tmp_path / 'tmp')


@pytest.mark.gpu
def test_launcher_with_the_reference_default_proximal_mutation(tmp_path):
    """base/train.py:32 defaults to -mut_type proximal: the Jacobian-scaled mutation runs batched on the device, fed by the
    per-actor device replay buffers the rollout kernel fills."""
    args = ['-frames', '9000', '-pop_size', '6', '-mut_type', 'proximal', '-test_ea']
    p = subprocess.run([sys.executable, os.path.join(ROOT, 'examples', 'train.py')] + args, cwd=tmp_path, capture_output=True, text=True,
                       timeout=1800)
    assert p.returncode == 0, p.stderr[-3000:]
    check_checkpoints(tmp_path / 'tmp')


@pytest.mark.gpu
def test_launcher_with_distillation_crossover_and_safe_mutation(tmp_path):
    """the reference's shipped operator set (SERL50 config.yaml: mut_type safe, distil_type fitness): Q-filtered distillation
    crossover and the safe mutation, both batched on the device."""
    args = ['-frames', '9000', '-pop_size', '8', '-mut_type', 'safe', '-use_distil', '-distil_type', 'fitness', '-test_ea']
    p = subprocess.run([sys.executable, os.path.join(ROOT, 'examples', 'train.py')] + args, cwd=tmp_path, capture_output=True, text=True,
                       timeout=1800)
    assert p.returncode == 0, p.stderr[-3000:]
    pop = torch.load(os.path.join(tmp_path, 'tmp', 'evo_nets.pkl'), weights_only=False)
    assert sorted(pop) == ['actor_%d' % i for i in range(8)]
    assert all(torch.isfinite(v).all() for v in pop['actor_3'].values())


def test_proximal_default_of_train_py_is_kept():
    """base/train.py's CLI default is -mut_type proximal: implemented (serl_b200/evo_prox.py), so Parameters keeps it."""
    import types
    from serl_b200.parameters import Parameters
    cwd = os.getcwd()
    os.chdir('/tmp')
    try:
        a = Parameters(types.SimpleNamespace(mut_type='proximal', pop_size=4))
    finally:
        os.chdir(cwd)
    assert a.mut_type == 'proximal'
