"""GPU: paacb_policy_forward (conv/fc implicit GEMMs, heads, softmax, sampling) against the oracle."""
import numpy as np
import pytest
import torch

from oracle import network, update
from util import assert_close
import gpu_util as G

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize('arch,A,b', [('NIPS', 4, 1), ('NIPS', 6, 33), ('NATURE', 6, 1), ('NATURE', 4, 7),
                                      ('NATURE', 6, 160), ('NATURE', 18, 129), ('NIPS', 18, 160), ('NIPS', 9, 37), ('NIPS', 2, 65)])
def test_forward_vs_oracle(arch, A, b):
    net = G.make_net(arch, A, seed=3)
    params = network.unflatten_params(net.get_params(), arch, A)
    ref0 = network.init_params(arch, A, 3)
    for k in params:
        assert (params[k] == ref0[k]).all(), 'init differs from the oracle init for ' + k
    rng = np.random.RandomState(b)
    states = rng.randint(0, 256, (b, 84, 84, 4)).astype(np.uint8)
    u = rng.random_sample(b).astype(np.float32)
    out = G.forward(net, states, u)
    ref = network.forward(params, states, arch, keep=True)
    acts = G.layer_acts(net, out['ws'], b)
    for i, a in enumerate(ref['acts']):
        assert_close(acts[i], a.numpy(), 1e-4, 'conv%d activation' % (i + 1))
    assert_close(acts[-1], ref['h'].numpy(), 1e-4, 'hidden fc')
    pi, v = out['pi'].cpu().numpy(), out['v'].cpu().numpy()
    assert_close(pi, ref['pi'].numpy(), 1e-4, 'pi')
    assert_close(v, ref['v'].numpy(), 1e-4, 'v')
    assert np.abs(pi.sum(1) - 1).max() < 1e-5
    # sampling: bit-exact action indices given the same uniforms and the GPU's own pi
    want = update.sample_actions(pi, u)
    got = out['actions'].cpu().numpy()
    assert (got == want).all()
    assert (out['onehot'].cpu().numpy() == np.eye(A, dtype=np.float32)[want]).all()


def test_sampling_edges_and_distribution():
    A = 6
    net = G.make_net('NIPS', A)
    b = 4096
    states = np.zeros((b, 84, 84, 4), np.uint8)          # identical inputs -> identical pi for every row
    rng = np.random.RandomState(0)
    u = rng.random_sample(b).astype(np.float32)
    u[:3] = [0.0, np.nextafter(np.float32(1), np.float32(0)), 0.5]
    out = G.forward(net, states, u)
    pi = out['pi'].cpu().numpy()
    a = out['actions'].cpu().numpy()
    assert a[0] == 0 and a[1] == A - 1 and (a == update.sample_actions(pi, u)).all()
    freq = np.bincount(a, minlength=A) / b
    assert np.abs(freq - pi[0]).max() < 0.03


def test_session_shim_and_choose_next_actions():
    from paac_b200.paac import PAACLearner
    from paac_b200.session import Session
    A = 4
    net = G.make_net('NATURE', A)
    states = np.random.RandomState(1).randint(0, 256, (5, 84, 84, 4)).astype(np.uint8)
    v, pi = Session().run([net.output_layer_v, net.output_layer_pi], feed_dict={net.input_ph: states})
    ref = network.forward(network.unflatten_params(net.get_params(), 'NATURE', A), states, 'NATURE')
    assert_close(pi, ref['pi'].numpy(), 1e-4); assert_close(v, ref['v'].numpy(), 1e-4)
    onehot, v2, pi2 = PAACLearner.choose_next_actions(net, A, states, None)
    assert onehot.shape == (5, A) and (onehot.sum(1) == 1).all() and np.array_equal(v2, v) and np.array_equal(pi2, pi)
