"""GPU: the tcgen05 tensor-core paths against the oracle.  PAACB_MATH_BF16X3 (bf16-split operands, TMA-fed
patch-resident implicit GEMMs; Nature architecture) and PAACB_MATH_TF32X3 are parity modes and meet the 1e-4 bar
(scaled max error, see util.py); plain TF32 rounds operands to 11 bits and is held to 3e-3 -- a speed mode only."""
import numpy as np
import pytest
import torch

from oracle import network, update
from paac_b200.engine import RolloutEngine
from util import assert_close, rel_err
import gpu_util as G

pytestmark = pytest.mark.gpu

TOL = {'bf16x3': 1e-4, 'tf32x3': 1e-4, 'tf32': 3e-3}
MODES = ['bf16x3', 'tf32x3', 'tf32']


def skip_unsupported(math, arch):
    """every tensor-core mode covers both architectures since round 2 (NIPS: 64-byte units, SWIZZLE_64B variants)"""


@pytest.mark.parametrize('math', MODES)
@pytest.mark.parametrize('arch,A,b', [('NATURE', 6, 1), ('NATURE', 6, 130), ('NIPS', 4, 33), ('NIPS', 6, 300), ('NATURE', 18, 517),
                                      ('NIPS', 9, 45), ('NIPS', 18, 101)])
def test_forward_tc_vs_oracle(math, arch, A, b):
    skip_unsupported(math, arch)
    net = G.make_net(arch, A, seed=3, math=math)
    params = network.unflatten_params(net.get_params(), arch, A)
    rng = np.random.RandomState(b)
    states = rng.randint(0, 256, (b, 84, 84, 4)).astype(np.uint8)
    out = G.forward(net, states)
    ref = network.forward(params, states, arch, dtype=torch.float64, keep=True)
    acts = G.layer_acts(net, out['ws'], b)
    for i, a in enumerate(ref['acts']):
        assert_close(acts[i], a.numpy(), TOL[math], 'conv%d activation' % (i + 1))
    assert_close(acts[-1], ref['h'].numpy(), TOL[math], 'hidden fc')
    assert_close(out['pi'].cpu().numpy(), ref['pi'].numpy(), TOL[math], 'pi')
    assert_close(out['v'].cpu().numpy(), ref['v'].numpy(), TOL[math], 'v')


@pytest.mark.parametrize('math', MODES)
# b = 129, 257, 130: the heads backward's last 128-sample CTA holds 1 or 2 samples
@pytest.mark.parametrize('arch,A,b', [('NATURE', 6, 5), ('NATURE', 6, 160), ('NIPS', 4, 97), ('NIPS', 6, 160), ('NATURE', 4, 1111),
                                      ('NIPS', 9, 129), ('NIPS', 18, 257), ('NATURE', 18, 130)])
def test_backward_tc_vs_autograd(math, arch, A, b):
    """Gradients (and every layer's dZ) against fp64 autograd whose ReLU masks are the GPU's own activations
    (oracle.network.masked_loss_and_grads): like-for-like, immune to a pre-activation rounding across zero."""
    skip_unsupported(math, arch)
    net = G.make_net(arch, A, seed=11, math=math)
    params = network.unflatten_params(net.get_params(), arch, A)
    rng = np.random.RandomState(b + A)
    states = rng.randint(0, 256, (b, 84, 84, 4)).astype(np.uint8)
    acts = rng.randint(0, A, b)
    adv = rng.randn(b).astype(np.float32); tgt = rng.randn(b).astype(np.float32)
    fwd = G.forward(net, states)
    masks = [x > 0 for x in G.layer_acts(net, fwd['ws'], b)]
    g64, dzs, f64 = network.masked_loss_and_grads(params, states, acts, adv, tgt, 0.02, arch, A, masks)
    _, dz, dv = network.closed_form_head_grads(f64['logits'], f64['v'], acts, adv, tgt, np.float32(0.02))
    flat, bws = G.backward(net, fwd, dz, dv)
    got = network.unflatten_params(flat, arch, A)
    for name, _, _ in network.param_specs(arch, A):
        assert_close(got[name], g64[name], TOL[math], name)
    for i, (d, got_dz) in enumerate(zip(dzs, G.layer_acts(net, bws, b))):
        assert_close(got_dz.reshape(d.shape), d, TOL[math], 'dZ of layer %d' % i)


def test_auto_math_is_bf16x3_for_both_architectures():
    for arch in ('NIPS', 'NATURE'):
        net = G.make_net(arch, 4, seed=3, math='auto')
        assert net.math == 'bf16x3' and net._lib.paacb_get_math(net.ctx) == 3


# T = 12 and 9: the loss kernel's warps take more than one time step each
@pytest.mark.parametrize('arch,math,A,T', [('NATURE', 'bf16x3', 6, 5), ('NATURE', 'tf32x3', 6, 5), ('NIPS', 'bf16x3', 6, 5),
                                          ('NIPS', 'bf16x3', 9, 12), ('NATURE', 'bf16x3', 18, 9)],
                         ids=['NATURE-bf16x3', 'NATURE-tf32x3', 'NIPS-bf16x3', 'NIPS-bf16x3-A9-T12', 'NATURE-bf16x3-A18-T9'])
def test_engine_update_tc_vs_oracle_composite(arch, math, A, T):
    N = 16
    net = G.make_net(arch, A, seed=5, math=math)
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
    eng.update(0.0224)
    torch.cuda.synchronize()
    params = network.unflatten_params(p0, arch, A)
    B = T * N
    acts = eng.actions.cpu().numpy().reshape(-1)
    y, adv = update.nstep_returns(rewards, over, eng.values.cpu().numpy(), eng.boot_v.cpu().numpy(), 0.99)
    loss, _, _ = network.loss_and_grads(params, states[:T].reshape(B, 84, 84, 4), acts, adv.reshape(-1), y.reshape(-1),
                                        np.float32(0.02), arch, A)
    assert abs(eng.loss.item() - loss) <= 1e-4 * max(1, abs(loss))
    masks = [x > 0 for x in G.layer_acts(net, eng.fwd_ws, B)]
    grads, _, _ = network.masked_loss_and_grads(params, states[:T].reshape(B, 84, 84, 4), acts, adv.reshape(-1), y.reshape(-1),
                                                np.float32(0.02), arch, A, masks)
    specs = network.param_specs(arch, A)
    clipped, norm = update.clip_by_global_norm([grads[n] for n, _, _ in specs], 3.0)
    assert abs(eng.norm.item() - float(norm)) <= 1e-4 * float(norm)
    new = {}
    for (n, s, _), gc in zip(specs, clipped):
        new[n], _, _ = update.rmsprop_apply(params[n], np.ones(s, np.float32), np.zeros(s, np.float32), gc, 0.0224, 0.99, 0.1)
    want = network.flatten_params(new, arch, A)
    got = net.get_params()
    assert_close(got, want, 1e-5, 'post-RMSProp weights')
    assert_close(got - p0, want - p0, 2e-3, 'weight delta')


def test_sliced_act_observe_equals_whole_batch():
    """RolloutEngine.act / observe_frames on contiguous environment slices (what the pipelined end-to-end loop issues on
    two streams) produce the same actions, values and states as the whole-batch calls."""
    arch, A, N, T = 'NATURE', 6, 24, 2
    rng = np.random.RandomState(7)
    s0 = rng.randint(0, 256, (N, 84, 84, 4)).astype(np.uint8)
    frames = G.dev(rng.randint(0, 256, (T, N, 1, 2, 210, 160)).astype(np.uint8))
    rew = G.dev(rng.choice([-1.0, 0.0, 1.0], size=(T, N)).astype(np.float32))
    over = G.dev(np.zeros((T, N), np.float32))
    outs = []
    for slices in ([(0, N)], [(0, 8), (8, 24)]):
        net = G.make_net(arch, A, seed=5, math='bf16x3')
        eng = RolloutEngine(net, N, T, seed=9)
        eng.state(0).copy_(G.dev(s0))
        eng.draw_uniforms()
        for t in range(T):
            for lo, hi in slices:
                eng.act(t, lo, hi)
            for lo, hi in slices:
                eng.observe_frames(t, frames[t, lo].data_ptr(), 1, None, rew[t], over[t], lo, hi)
        torch.cuda.synchronize()
        outs.append((eng.actions.cpu().numpy(), eng.values.cpu().numpy(), eng.get_states().cpu().numpy(), eng.rewards.cpu().numpy()))
    assert np.array_equal(outs[0][0], outs[1][0]) and np.array_equal(outs[0][2], outs[1][2])
    assert np.array_equal(outs[0][3], outs[1][3])
    assert_close(outs[1][1], outs[0][1], 1e-6, 'values of sliced vs whole-batch forward')


@pytest.mark.parametrize('math', ['bf16x3', 'tf32x3', 'fp32'])
def test_training_forward_schedules_are_bit_identical(math):
    """The training forward of PAAC is the concatenation of the acting forwards under unchanged parameters (paac.py:92,112,151).
    'batched' (one forward over T*N samples in update()), 'stepwise' (paacb_policy_forward_at per step / slice) and 'reuse'
    (the acting forward writes the training workspace) must leave the SAME BITS in the activation workspace, pi and v, and
    the same update (gradient sums use atomics, so the post-update weights are compared to rounding)."""
    arch, A, N, T = 'NATURE', 6, 40, 3
    rng = np.random.RandomState(11)
    states = rng.randint(0, 256, (T + 1, N, 84, 84, 4)).astype(np.uint8)
    rewards = rng.choice([-1.0, 0.0, 1.0], size=(T, N)).astype(np.float32)
    over = (rng.random_sample((T, N)) < 0.2).astype(np.float32)
    res = {}
    for mode in ('batched', 'stepwise', 'reuse'):
        net = G.make_net(arch, A, seed=5, math=math)
        eng = RolloutEngine(net, N, T, seed=9, train_forward=mode)
        eng.set_states(G.dev(states))
        eng.draw_uniforms()
        for t in range(T):
            eng.act(t, 0, 16)
            eng.act(t, 16, N)
            if mode == 'stepwise' and t != 1:                # step 1 is left to update(); step 2 is issued in two slices
                if t == 2:
                    eng.train_forward_step(t, 0, 24)
                    eng.train_forward_step(t, 24, N)
                else:
                    eng.train_forward_step(t)
        eng.rewards.copy_(G.dev(rewards)); eng.over.copy_(G.dev(over))
        eng.update(0.0224)
        torch.cuda.synchronize()
        res[mode] = dict(ws=eng.fwd_ws.view(torch.int32).cpu().numpy().copy(), pi=eng.pi.cpu().numpy().copy(),
                         v=eng.v.cpu().numpy().copy(), values=eng.values.cpu().numpy().copy(),
                         actions=eng.actions.cpu().numpy().copy(), y=eng.y.cpu().numpy().copy(),
                         loss=eng.loss.item(), params=net.get_params())
    ref = res['batched']
    for mode in ('stepwise', 'reuse'):
        r = res[mode]
        assert np.array_equal(r['actions'], ref['actions']), mode
        assert np.array_equal(r['ws'], ref['ws']), mode + ': activation workspace differs'
        assert np.array_equal(r['pi'].view(np.int32), ref['pi'].view(np.int32)), mode
        assert np.array_equal(r['v'].view(np.int32), ref['v'].view(np.int32)), mode
        assert np.array_equal(r['values'].view(np.int32), ref['values'].view(np.int32)), mode
        assert np.array_equal(r['y'].view(np.int32), ref['y'].view(np.int32)), mode
        assert abs(r['loss'] - ref['loss']) <= 1e-6 * max(1.0, abs(ref['loss']))
        assert_close(r['params'], ref['params'], 1e-6, mode + ': post-update weights')


def test_cached_weight_images_follow_the_parameters():
    """The bf16x3 forward reuses the operand images of the weights between calls (paacb_params_changed contract):
    after set_params() and after paacb_clip_rmsprop the next forward must see the NEW parameters."""
    arch, A, N, T = 'NATURE', 6, 8, 2
    rng = np.random.RandomState(3)
    states = G.dev(rng.randint(0, 256, (N, 84, 84, 4)).astype(np.uint8))

    def fwd(net):
        pi = torch.empty((N, A), device='cuda'); v = torch.empty((N,), device='cuda')
        ws = torch.empty((net.workspace_floats(N),), device='cuda')
        net.forward(states, pi, v, ws)
        torch.cuda.synchronize()
        return pi.cpu().numpy(), v.cpu().numpy()

    net = G.make_net(arch, A, seed=5, math='bf16x3')
    other = G.make_net(arch, A, seed=6, math='bf16x3')
    pi0, v0 = fwd(net)
    net.set_params(other.get_params())                      # host write -> params_changed()
    pi1, v1 = fwd(net)
    pi_o, v_o = fwd(other)
    assert np.array_equal(pi1, pi_o) and np.array_equal(v1, v_o)
    assert not np.array_equal(v0, v1)
    # an update through the library refreshes the images in-stream
    eng = RolloutEngine(net, N, T, seed=9)
    eng.set_states(G.dev(rng.randint(0, 256, (T + 1, N, 84, 84, 4)).astype(np.uint8)))
    eng.draw_uniforms()
    for t in range(T):
        eng.act(t)
    eng.rewards.fill_(1.0)
    eng.update(0.0224)
    pi2, v2 = fwd(net)
    fresh = G.make_net(arch, A, seed=1, math='bf16x3')
    fresh.set_params(net.get_params())
    pi_f, v_f = fwd(fresh)
    assert np.array_equal(pi2, pi_f) and np.array_equal(v2, v_f)
    assert not np.array_equal(v1, v2)


@pytest.mark.parametrize('arch', ['NATURE', 'NIPS'])
def test_forward_bits_do_not_depend_on_slices_or_streams(arch):
    """The bf16x3 forward of a batch leaves the same bits in the activation workspace, pi and v whether it is issued whole or
    as ragged slices of one workspace (paacb_policy_forward_at), also after new parameters, and when the forwards of two
    batches alternate on two streams."""
    A = 6
    net = G.make_net(arch, A, seed=13, math='bf16x3')
    gen = torch.Generator(device='cuda'); gen.manual_seed(6)
    states = torch.randint(0, 256, (600, 84, 84, 4), dtype=torch.uint8, device='cuda', generator=gen)

    def run(s):
        b = s.shape[0]
        pi = torch.full((b, A), -1.0, device='cuda'); v = torch.full((b,), -1.0, device='cuda')
        ws = torch.zeros((net.workspace_floats(b),), device='cuda')
        net.forward(s, pi, v, ws)
        torch.cuda.synchronize()
        return ws.view(torch.int32).clone(), pi, v

    def sliced():
        pi = torch.zeros((600, A), device='cuda'); v = torch.zeros((600,), device='cuda')
        ws = torch.zeros((net.workspace_floats(600),), device='cuda')
        for lo, hi in ((0, 250), (250, 251), (251, 600)):
            net.forward(states[lo:hi], pi[lo:hi], v[lo:hi], ws, ws_capacity=600, ws_first=lo)
        torch.cuda.synchronize()
        return ws.view(torch.int32).clone(), pi, v

    whole = run(states)
    for a, b in zip(whole, sliced()):
        assert torch.equal(a, b)
    # new parameters: the cached operand images are refreshed
    net.set_params(net.get_params() * np.float32(0.5))
    whole_new, sliced_new = run(states), sliced()
    for a, b in zip(whole_new, sliced_new):
        assert torch.equal(a, b)
    assert not torch.equal(sliced_new[2], whole[2])

    sa = torch.randint(0, 256, (2000, 84, 84, 4), dtype=torch.uint8, device='cuda', generator=gen)
    sb = torch.randint(0, 256, (1500, 84, 84, 4), dtype=torch.uint8, device='cuda', generator=gen)
    ra, rb = run(sa), run(sb)
    outs = []
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    for s in (sa, sb):
        b = s.shape[0]
        pi = torch.zeros((b, A), device='cuda'); v = torch.zeros((b,), device='cuda')
        ws = torch.zeros((net.workspace_floats(b),), device='cuda')
        outs.append((ws, pi, v))
    torch.cuda.synchronize()
    for rep in range(3):
        for st, s, (ws, pi, v) in zip(streams, (sa, sb), outs):
            with torch.cuda.stream(st):
                net.forward(s, pi, v, ws)
    torch.cuda.synchronize()
    for ref, (ws, pi, v) in zip((ra, rb), outs):
        assert torch.equal(ref[0], ws.view(torch.int32)) and torch.equal(ref[1], pi) and torch.equal(ref[2], v)


def test_sliced_bootstrap_equals_whole_batch():
    """RolloutEngine.bootstrap(lo, hi) per environment slice (what the end-to-end loop issues as each slice's last frames
    arrive) leaves the same V(s_T), loss and update as the whole-batch bootstrap inside update()."""
    arch, A, N, T = 'NATURE', 6, 24, 2
    rng = np.random.RandomState(13)
    states = rng.randint(0, 256, (T + 1, N, 84, 84, 4)).astype(np.uint8)
    rewards = rng.choice([-1.0, 0.0, 1.0], size=(T, N)).astype(np.float32)
    outs = []
    for sliced in (False, True):
        net = G.make_net(arch, A, seed=5, math='bf16x3')
        eng = RolloutEngine(net, N, T, seed=9)
        eng.set_states(G.dev(states))
        eng.draw_uniforms()
        for t in range(T):
            eng.act(t)
        eng.rewards.copy_(G.dev(rewards))
        if sliced:
            eng.bootstrap(8, 24)          # slice 0 is left to update()
        eng.update(0.0224)
        torch.cuda.synchronize()
        outs.append((eng.boot_v.cpu().numpy(), eng.y.cpu().numpy(), eng.loss.item(), net.get_params()))
    assert np.array_equal(outs[0][0].view(np.int32), outs[1][0].view(np.int32))
    assert np.array_equal(outs[0][1].view(np.int32), outs[1][1].view(np.int32))
    assert abs(outs[0][2] - outs[1][2]) <= 1e-6 * max(1.0, abs(outs[0][2]))
    assert_close(outs[1][3], outs[0][3], 1e-6, 'post-update weights')


@pytest.mark.parametrize('b', [1, 2, 3, 37, 148 * 2 + 1, 1111])
def test_conv3_packed_tiles_vs_oracle(b):
    """conv3's forward with two whole samples per tile (Geo<G_FWD3P>: three patch copies, row groups at a 9-unit stride), run
    into a slice of a larger workspace, against the fp64 oracle: every layer's activations, pi and v.  Odd batches
    (zero-filled half tile), one tile, more tiles than SMs; samples outside the slice stay untouched."""
    A = 6
    net = G.make_net('NATURE', A, seed=21, math='bf16x3')
    params = network.unflatten_params(net.get_params(), 'NATURE', A)
    gen = torch.Generator(device='cuda'); gen.manual_seed(100 + b)
    states = torch.randint(0, 256, (b, 84, 84, 4), dtype=torch.uint8, device='cuda', generator=gen)
    cap, first = b + 5, 3
    pi = torch.full((b, A), -1.0, device='cuda'); v = torch.full((b,), -1.0, device='cuda')
    ws = torch.zeros((net.workspace_floats(cap),), device='cuda')
    net.forward(states, pi, v, ws, ws_capacity=cap, ws_first=first)
    torch.cuda.synchronize()
    ref = network.forward(params, states.cpu().numpy(), 'NATURE', dtype=torch.float64, keep=True)
    acts = G.layer_acts(net, ws, cap)
    for i, want in enumerate(ref['acts'] + [ref['h']]):
        name = 'conv%d activation' % (i + 1) if i < len(ref['acts']) else 'hidden fc'
        assert_close(acts[i][first:first + b], want.numpy(), TOL['bf16x3'], name)
        assert not acts[i][:first].any() and not acts[i][first + b:].any(), name + ': outside the slice'
    assert_close(pi.cpu().numpy(), ref['pi'].numpy(), TOL['bf16x3'], 'pi')
    assert_close(v.cpu().numpy(), ref['v'].numpy(), TOL['bf16x3'], 'v')
