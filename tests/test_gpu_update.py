"""GPU: returns+loss gradient, backward, clip+RMSProp and the whole update against the oracle and against the
outputs of the reference's shipped TF graph (tests/golden/tf_graph_nips.npz)."""
import os

import numpy as np
import pytest
import torch

from oracle import network, update
from oracle.make_golden import gen_train_batch
from paac_b200 import _lib
from paac_b200.engine import RolloutEngine
from util import assert_close, rel_err
import gpu_util as G

pytestmark = pytest.mark.gpu


# T > 8: the kernel's 8 warps each take several time steps (t = w, w + 8, ...) and reload pi, v and the action for all but
# the first; T = 64 is the kernel's limit (kLossMaxT)
@pytest.mark.parametrize('T,N,A,gamma', [(5, 37, 6, 0.99), (1, 1, 4, 0.99), (5, 256, 18, 0.99), (3, 130, 6, 0.99),
                                         (8, 33, 9, 0.99), (9, 31, 18, 0.99), (16, 100, 2, 0.99), (17, 37, 3, 0.99),
                                         (64, 65, 9, 0.99), (9, 31, 18, 0.0), (17, 37, 3, 1.0)],
                         ids=['5-37-6', '1-1-4', '5-256-18', '3-130-6', '8-33-9', '9-31-18', '16-100-2', '17-37-3', '64-65-9',
                              '9-31-18-gamma0', '17-37-3-gamma1'])
def test_returns_loss_grad_vs_oracle(T, N, A, gamma):
    net = G.make_net('NIPS', A)
    rng = np.random.RandomState(T * 1000 + N)
    rewards = rng.choice([-3.0, -1.0, 0.0, 0.5, 1.0, 7.0], size=(T, N)).astype(np.float32)
    over = (rng.random_sample((T, N)) < 0.2).astype(np.float32)
    values = rng.randn(T, N).astype(np.float32)
    boot = rng.randn(N).astype(np.float32)
    actions = rng.randint(0, A, T * N).astype(np.int32)
    logits = rng.randn(T * N, A) * 2
    logits[0, :] = [-100] * (A - 1) + [50]                      # a saturated policy row
    pi = np.exp(logits - logits.max(1, keepdims=True)); pi = (pi / pi.sum(1, keepdims=True)).astype(np.float32)
    v = rng.randn(T * N).astype(np.float32)
    out = G.returns_loss_grad(net, rewards, over, values, boot, actions, pi, v, gamma, 0.02)
    y, adv = update.nstep_returns(rewards, over, values, boot, gamma)
    assert np.array_equal(out['y'], y.reshape(-1)) and np.array_equal(out['adv'], adv.reshape(-1))   # f64 recurrence -> f32
    # loss / gradients: feed pi through the exact-epsilon closed form in float64 (SURVEY App. C)
    z = np.log(pi.astype(np.float64) + 1e-300)
    loss, dz, dvv = network.closed_form_head_grads(z, v, actions, adv.reshape(-1), y.reshape(-1), np.float32(0.02))
    assert abs(out['loss'][0] - loss) <= 1e-5 * max(1.0, abs(loss))
    assert_close(out['dlogits'], dz, 1e-5, 'dlogits')
    assert_close(out['dv'], dvv, 1e-6, 'dv')


@pytest.mark.parametrize('arch,A,b', [('NIPS', 4, 3), ('NATURE', 6, 5), ('NATURE', 6, 160), ('NIPS', 18, 97), ('NATURE', 4, 40),
                                      ('NATURE', 6, 1111)])
def test_backward_vs_autograd(arch, A, b):
    net = G.make_net(arch, A, seed=11)
    params = network.unflatten_params(net.get_params(), arch, A)
    rng = np.random.RandomState(b + A)
    states = rng.randint(0, 256, (b, 84, 84, 4)).astype(np.uint8)
    acts = rng.randint(0, A, b)
    adv = rng.randn(b).astype(np.float32); tgt = rng.randn(b).astype(np.float32)
    fwd = G.forward(net, states)
    # fp64 autograd with the GPU's own ReLU masks (see oracle.network.masked_loss_and_grads)
    masks = [x > 0 for x in G.layer_acts(net, fwd['ws'], b)]
    g64, dzs, f64 = network.masked_loss_and_grads(params, states, acts, adv, tgt, 0.02, arch, A, masks)
    _, dz, dv = network.closed_form_head_grads(f64['logits'], f64['v'], acts, adv, tgt, np.float32(0.02))
    flat, bws = G.backward(net, fwd, dz, dv)
    got = network.unflatten_params(flat, arch, A)
    for name, _, _ in network.param_specs(arch, A):
        assert_close(got[name], g64[name], 1e-4, name)
    off = 0
    for i, d in enumerate(dzs):
        assert_close(bws[off:off + d.size].cpu().numpy().reshape(d.shape), d, 1e-4, 'dZ of layer %d' % i)
        off += d.size


@pytest.mark.parametrize('arch,math', [('NATURE', 'bf16x3'), ('NATURE', 'tf32x3'), ('NIPS', 'fp32')])
def test_backward_parts_equal_whole(arch, math):
    """paacb_backward_part(TAIL) leaves d_grads[tail_offset:] final (it can be all-reduced while the rest runs);
    TAIL followed by HEAD equals paacb_backward (gradient sums use atomics: compared to rounding)."""
    A, b = 6, 50
    net = G.make_net(arch, A, seed=11, math=math)
    rng = np.random.RandomState(5)
    states = rng.randint(0, 256, (b, 84, 84, 4)).astype(np.uint8)
    fwd = G.forward(net, states)
    dl = G.dev((rng.randn(b, A) * 0.01).astype(np.float32)); dv = G.dev((rng.randn(b) * 0.01).astype(np.float32))
    whole, _ = G.backward(net, fwd, dl.cpu().numpy(), dv.cpu().numpy())
    bws = torch.zeros((int(net._lib.paacb_backward_workspace_floats(net.ctx, b)),), dtype=torch.float32, device='cuda')
    grads = torch.full((net.param_count,), 7.0, dtype=torch.float32, device='cuda')
    p = _lib.ptr
    tail = int(net._lib.paacb_grad_tail_offset(net.ctx))
    assert 0 < tail < net.param_count and net.param_count - tail > 0.9 * net.param_count
    _lib.check(net._lib.paacb_backward_part(net.ctx, p(net.params), p(fwd['states']), b, p(fwd['ws']), p(dl), p(dv), p(bws),
                                            p(grads), _lib.BWD_TAIL, G.stream()), 'tail')
    torch.cuda.synchronize()
    after_tail = grads.cpu().numpy()
    assert_close(after_tail[tail:], whole[tail:], 1e-6, 'tail of the gradient after PAACB_BWD_TAIL')
    _lib.check(net._lib.paacb_backward_part(net.ctx, p(net.params), p(fwd['states']), b, p(fwd['ws']), p(dl), p(dv), p(bws),
                                            p(grads), _lib.BWD_HEAD, G.stream()), 'head')
    torch.cuda.synchronize()
    both = grads.cpu().numpy()
    assert np.array_equal(both[tail:], after_tail[tail:])          # HEAD does not touch the tail
    assert_close(both, whole, 1e-6, 'TAIL + HEAD vs paacb_backward')


@pytest.mark.parametrize('clip_type,gscale', [(_lib.CLIP_GLOBAL, 1.0), (_lib.CLIP_GLOBAL, 0.125), (_lib.CLIP_IGNORE, 1.0)])
def test_clip_rmsprop_vs_oracle(clip_type, gscale):
    net = G.make_net('NIPS', 6)                  # P = 677,943: not a multiple of 4 -> exercises the scalar tail
    P = net.param_count
    assert P % 4 != 0
    rng = np.random.RandomState(2)
    params = rng.randn(P).astype(np.float32) * 0.05
    ms = (1 + 0.1 * rng.rand(P)).astype(np.float32); mom = (0.01 * rng.randn(P)).astype(np.float32)
    grads = (rng.randn(P) * 0.05).astype(np.float32)
    for momentum in (0.0, 0.9):
        p2, ms2, mom2, norm = G.clip_rmsprop(net, params, ms, mom, grads, gscale, 0.0224, 0.99, 0.1, momentum, 3.0, clip_type)
        g = grads * np.float32(gscale)
        want_norm = float(np.sqrt(np.sum(g.astype(np.float64) ** 2)))
        assert abs(norm - want_norm) <= 1e-5 * want_norm
        if clip_type == _lib.CLIP_GLOBAL:
            (gc,), _ = update.clip_by_global_norm([g], 3.0)
        else:
            gc = g
        wp, wms, wmom = update.rmsprop_apply(params, ms, mom, gc, 0.0224, 0.99, 0.1, momentum)
        assert_close(ms2, wms, 1e-6, 'ms'); assert_close(mom2, wmom, 1e-5, 'mom'); assert_close(p2, wp, 1e-6, 'params')
        assert_close(p2 - params, wp - params, 1e-4, 'delta')
    rc = net._lib.paacb_clip_rmsprop(net.ctx, None, None, None, None, 1.0, 0.1, 0.99, 0.1, 0.0, 3.0, 1, None, None, None)
    assert rc == -1


@pytest.mark.parametrize('arch', ['NIPS', 'NATURE'])
def test_fused_optimizer_equals_two_pass_bitwise(arch, monkeypatch):
    """The cooperative one-launch optimizer (gradient held in registers across a grid barrier) and the two-launch version
    (sumsq partials, then update) are the same arithmetic in the same order: identical bits, over repeated launches (the
    barrier counter is monotonic across launches)."""
    rng = np.random.RandomState(4)
    outs = {}
    for two_pass in ('0', '1'):
        monkeypatch.setenv('PAACB_OPT_TWO_PASS', two_pass)
        net = G.make_net(arch, 6)
        P = net.param_count
        params = (rng.randn(P) * 0.05).astype(np.float32) if two_pass == '0' else outs['in'][0]
        ms = (1 + 0.1 * rng.rand(P)).astype(np.float32) if two_pass == '0' else outs['in'][1]
        mom = (0.01 * rng.randn(P)).astype(np.float32) if two_pass == '0' else outs['in'][2]
        grads = [(rng.randn(P) * s).astype(np.float32) for s in (0.05, 1e-4, 3.0)] if two_pass == '0' else outs['in'][3]
        outs['in'] = (params, ms, mom, grads)
        st = (params, ms, mom)
        res = []
        for g in grads:
            p2, ms2, mom2, norm = G.clip_rmsprop(net, st[0], st[1], st[2], g, 0.125, 0.0224, 0.99, 0.1, 0.9, 3.0, _lib.CLIP_GLOBAL)
            st = (p2, ms2, mom2)
            res.append((p2, ms2, mom2, norm))
        outs[two_pass] = res
    for a, b in zip(outs['0'], outs['1']):
        for x, y in zip(a[:3], b[:3]):
            assert np.array_equal(x.view(np.int32), y.view(np.int32))
        assert a[3] == b[3]


@pytest.mark.parametrize('math', ['fp32', 'tf32x3', 'bf16x3'])
def test_two_updates_match_reference_tf_graph(golden_dir, math):
    """The same two train steps the reference's shipped graph was evaluated on (NIPS, A=4, b=12), in the fp32 anchor AND in
    both tensor-core parity modes: the reference's own serialized graph pins every arithmetic path directly."""
    g = np.load(os.path.join(golden_dir, 'tf_graph_nips.npz'))
    A, b = int(g['A']), int(g['b'])
    net = G.make_net('NIPS', A, seed=int(g['wseed']), math=math)
    eng = RolloutEngine(net, n_envs=b, t_max=1, gamma=1.0, rho=0.99, eps=0.1, clip_norm=3.0, clip_norm_type='global')
    for step in range(2):
        states, acts, adv, tgt = gen_train_batch(int(g['bseed']) + step, b, A)
        # make paacb_returns_loss_grad reproduce the fed placeholders: gamma = 1, r = 0, no terminal => y = V(s_T) := tgt,
        # adv = y - values with values := tgt - adv.  The bootstrap forward is overwritten by injecting boot_v.
        eng.state(0).copy_(G.dev(states)); eng.state(1).copy_(G.dev(states))
        eng.actions.copy_(G.dev(acts.reshape(1, b), torch.int32))
        eng.rewards.zero_(); eng.over.zero_()
        eng.values.copy_(G.dev((tgt - adv).reshape(1, b)))
        p = _lib.ptr
        flat_states = eng.flat_states
        net.forward(flat_states, eng.pi, eng.v, eng.fwd_ws)
        eng.boot_v.copy_(G.dev(tgt))
        _lib.check(eng.lib.paacb_returns_loss_grad(eng.ctx, p(eng.rewards), p(eng.over), p(eng.values), p(eng.boot_v),
                                                   p(eng.actions), p(eng.pi), p(eng.v), 1, b, 1.0, 0.02, p(eng.y), p(eng.adv),
                                                   p(eng.dlogits), p(eng.dv), p(eng.loss), eng._stream()))
        _lib.check(eng.lib.paacb_backward(eng.ctx, p(net.params), p(flat_states), b, p(eng.fwd_ws), p(eng.dlogits), p(eng.dv),
                                          p(eng.bwd_ws), p(eng.grads), eng._stream()))
        eng.apply(float(g['lr']))
        torch.cuda.synchronize()
        assert_close(eng.pi.cpu().numpy(), g['pi%d' % step], 1e-4, 'pi'); assert_close(eng.v.cpu().numpy(), g['v%d' % step], 1e-4, 'v')
        assert abs(eng.loss.item() - float(g['loss%d' % step])) <= 1e-4 * abs(float(g['loss%d' % step]))
        assert abs(eng.norm.item() - float(g['norm%d' % step])) <= 1e-4 * float(g['norm%d' % step])
        specs = network.param_specs('NIPS', A)
        gr = network.unflatten_params(eng.grads.cpu().numpy(), 'NIPS', A)
        sumsq = np.asarray([np.sum(gr[n].astype(np.float64) ** 2) for n, _, _ in specs])
        assert_close(sumsq, g['raw_sumsq%d' % step], 2e-4, 'raw grad sumsq')
        head = np.concatenate([gr[n].reshape(-1)[:64] for n, _, _ in specs])
        assert_close(head, g['raw_grad_head%d' % step], 1e-4, 'raw grad head')
        flat = net.get_params()
        assert_close(flat[::997], g['var_sample%d' % step], 1e-5, 'variables after ApplyRMSProp')


def test_engine_update_vs_oracle_composite():
    arch, A, N, T = 'NATURE', 6, 8, 5
    net = G.make_net(arch, A, seed=5)
    eng = RolloutEngine(net, N, T, seed=9)
    rng = np.random.RandomState(0)
    states = rng.randint(0, 256, (T + 1, N, 84, 84, 4)).astype(np.uint8)
    eng.set_states(G.dev(states))
    eng.draw_uniforms()
    for t in range(T):
        eng.act(t)
    rewards = rng.choice([-2.0, 0.0, 1.0], size=(T, N)).astype(np.float32)
    over = (rng.random_sample((T, N)) < 0.15).astype(np.float32)
    eng.rewards.copy_(G.dev(rewards)); eng.over.copy_(G.dev(over))
    p0 = net.get_params()
    lr = 0.0224
    eng.update(lr)
    torch.cuda.synchronize()
    # oracle composite (paac.py:105-165)
    params = network.unflatten_params(p0, arch, A)
    B = T * N
    vals = np.stack([network.forward(params, states[t], arch)['v'].numpy() for t in range(T)])
    assert_close(eng.values.cpu().numpy(), vals, 1e-4, 'acting values')
    acts = eng.actions.cpu().numpy().reshape(-1)
    boot = network.forward(params, states[T], arch)['v'].numpy()
    y, adv = update.nstep_returns(rewards, over, eng.values.cpu().numpy(), eng.boot_v.cpu().numpy(), 0.99)
    assert_close(eng.boot_v.cpu().numpy(), boot, 1e-4, 'bootstrap')
    assert np.array_equal(eng.y.cpu().numpy(), y.reshape(-1))
    loss, grads, _ = network.loss_and_grads(params, states[:T].reshape(B, 84, 84, 4), acts, adv.reshape(-1), y.reshape(-1),
                                            np.float32(0.02), arch, A)
    assert abs(eng.loss.item() - loss) <= 1e-4 * max(1, abs(loss))
    specs = network.param_specs(arch, A)
    clipped, norm = update.clip_by_global_norm([grads[n] for n, _, _ in specs], 3.0)
    assert abs(eng.norm.item() - float(norm)) <= 1e-4 * float(norm)
    new = {}
    for (n, s, _), gc in zip(specs, clipped):
        new[n], _, _ = update.rmsprop_apply(params[n], np.ones(s, np.float32), np.zeros(s, np.float32), gc, lr, 0.99, 0.1)
    want = network.flatten_params(new, arch, A)
    got = net.get_params()
    assert_close(got, want, 1e-5, 'post-RMSProp weights')
    assert_close(got - p0, want - p0, 2e-3, 'weight delta')
    # the rollout's last state is the next rollout's first (paac.py:99-112), without a copy: the halves flipped
    assert torch.equal(eng.state(0), G.dev(states[T]))
