"""GPU: configurations the default run never reaches -- rollouts longer than the loss kernel's limit, the exact boundary of
the inverse-CDF sampler, and the persistent conv weight-gradient kernels on a grid reduced by paacb_set_sm_reserve (what
every multi-GPU update runs)."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import network, update
from paac_b200 import _lib
from paac_b200.engine import RolloutEngine
from util import assert_close, rel_err
import gpu_util as G

pytestmark = pytest.mark.gpu

PAACB_EINVAL, PAACB_EUNSUPPORTED = -1, -3


def test_t_max_above_the_loss_kernel_limit_is_refused():
    A, T, N = 6, 65, 33
    net = G.make_net('NIPS', A)
    f = lambda *shape: torch.zeros(shape, device='cuda')
    y = torch.full((T * N,), 5.0, device='cuda')
    loss = torch.full((1,), 123.0, device='cuda')
    actions = torch.zeros((T * N,), dtype=torch.int32, device='cuda')
    p = _lib.ptr
    rc = net._lib.paacb_returns_loss_grad(net.ctx, p(f(T, N)), p(f(T, N)), p(f(T, N)), p(f(N)), p(actions), p(f(T * N, A)),
                                          p(f(T * N)), T, N, C.c_double(0.99), C.c_float(0.02), p(y), p(f(T * N)),
                                          p(f(T * N, A)), p(f(T * N)), p(loss), G.stream())
    torch.cuda.synchronize()
    assert rc == PAACB_EUNSUPPORTED and b'64' in net._lib.paacb_last_error()
    assert loss.item() == 123.0 and bool((y == 5.0).all())          # nothing was launched, not even the loss reset
    # the engine refuses such a rollout length before it allocates a buffer, rather than after the first rollout
    before = torch.cuda.memory_allocated()
    with pytest.raises(ValueError, match='64'):
        RolloutEngine(net, N, T)
    assert torch.cuda.memory_allocated() == before
    assert RolloutEngine(net, 4, 64).T == 64


@pytest.mark.parametrize('math', ['bf16x3', 'fp32'])
@pytest.mark.parametrize('arch,A', [('NIPS', 2), ('NATURE', 18)])
def test_sampling_at_the_cumulative_sums(arch, A, math):
    """The sampler takes the first j with u < c_j, strictly (c_j: fp32 running sum of pi in index order).  With uniforms
    injected exactly ON the running sums of the GPU's own pi, u = c_j must select j + 1 (or the next j whose sum is larger),
    bit for bit as oracle.update.sample_actions; u = 0 and the largest float below 1 are the two ends."""
    b = 61
    net = G.make_net(arch, A, seed=7, math=math)
    states = np.random.RandomState(A).randint(0, 256, (b, 84, 84, 4)).astype(np.uint8)
    pi = G.forward(net, states)['pi'].cpu().numpy()
    c = np.zeros((b, A - 1), np.float32)
    run = np.zeros(b, np.float32)
    for j in range(A - 1):
        run = (run + pi[:, j]).astype(np.float32)
        c[:, j] = run
    ends = np.where(np.arange(b) % 2 == 0, np.float32(0), np.nextafter(np.float32(1), np.float32(0))).astype(np.float32)
    for j in list(range(A - 1)) + ['ends']:
        u = ends if j == 'ends' else c[:, j]
        out = G.forward(net, states, u)
        assert np.array_equal(out['pi'].cpu().numpy().view(np.int32), pi.view(np.int32))      # the same pi as the sums above
        got = out['actions'].cpu().numpy()
        assert np.array_equal(got, update.sample_actions(pi, u)), 'u = c_%s' % j
        assert np.array_equal(out['onehot'].cpu().numpy(), np.eye(A, dtype=np.float32)[got])
        if j == 'ends':
            assert (got[0::2] == 0).all()                    # the initial weights give every action a share well above 2^-24
        else:
            nxt = c[:, j + 1] if j + 1 < A - 1 else np.full(b, np.inf, np.float32)
            strict = nxt > c[:, j]                           # the next bucket is not empty in fp32
            assert strict.sum() > b // 2 and (got[strict] == j + 1).all(), 'u = c_%d' % j


@pytest.mark.parametrize('arch', ['NATURE', 'NIPS'])
def test_conv_weight_gradients_with_reserved_sms(arch):
    """With paacb_set_sm_reserve(r) the persistent bf16x3 conv weight-gradient kernels run on S - r CTAs, each taking a
    contiguous range of ceil(stages / grid) stages (conv1: 2b stages, conv2: b, conv3: ceil(b / 2)).  b = S - r + 1 puts
    conv2 one stage past the grid (half of the CTAs get no stage); r = S - 1 runs every stage on one CTA through its two
    buffer slots.  The gradients must meet the fp64 arbiter, and at r = 8 (the multi-GPU engine's reserve) equal the r = 0
    result up to the order of the atomic adds.
    r = S - 1 is held to the arbiter only: its one CTA accumulates every stage in one tensor-memory sum, and the error of that
    sum grows with the number of stages (measured on a B200 at 1000 W, Nature: conv1's weight gradient at b = 141, i.e. 282
    stages on one CTA, is 7.8e-5 of scale from fp64 and 1.3e-5 from r = 0, against 8.5e-6 from fp64 at r = 0).  Its largest
    batch keeps one CTA's stage count below what each CTA accumulates in the benchmarked configuration (about 277 conv1
    stages at 4096 environments and t_max 5)."""
    S = torch.cuda.get_device_properties(0).multi_processor_count
    A = 6
    batches = {0: [1, 2, 37, S - 7, S + 1, 301], 8: [1, S - 7, 301], S - 1: [1, 2, 37]}
    rng = np.random.RandomState(17)
    data = {b: (rng.randint(0, 256, (b, 84, 84, 4)).astype(np.uint8), (rng.randn(b, A) * 0.01).astype(np.float32),
                (rng.randn(b) * 0.01).astype(np.float32)) for b in batches[0]}
    conv_names = [n for n, _, _ in network.param_specs(arch, A)][:2 * len(network.ARCH[arch]['convs'])]
    base = {}
    for r in batches:
        net = G.make_net(arch, A, seed=11, math='bf16x3')
        assert net._lib.paacb_set_sm_reserve(net.ctx, r) == 0
        tail = int(net._lib.paacb_grad_tail_offset(net.ctx))
        for b in batches[r]:
            states, dl, dv = data[b]
            fwd = G.forward(net, states)
            flat, _ = G.backward(net, fwd, dl, dv)
            want = G.fp64_masked_grads_cuda(arch, A, net.get_params(), fwd['states'], net.layer_tensors(fwd['ws'], b),
                                            G.dev(dl), G.dev(dv))
            got = network.unflatten_params(flat, arch, A)
            for name in conv_names:
                assert_close(got[name], want[name], 1e-4, '%s r=%d b=%d' % (name, r, b))
            if r == 0:
                base[b] = flat[:tail]
            elif r == 8:
                # the fp32 atomics of ~100 partial sums land in another order on every run (NIPS, b = 301: up to 1.04e-6 of
                # scale observed); a stage that no CTA runs moves the sum by about 1 / b of scale
                assert rel_err(flat[:tail], base[b]) <= 1e-5, 'r=%d b=%d against r=0' % (r, b)
            if r == 8 and b == S - r + 1:
                # the multi-GPU engine's sequence: PAACB_BWD_TAIL, then PAACB_BWD_HEAD (the conv layers) under the tail's all-reduce
                bws = torch.zeros((int(net._lib.paacb_backward_workspace_floats(net.ctx, b)),), device='cuda')
                grads = torch.full((net.param_count,), 7.0, device='cuda')
                dl_d, dv_d = G.dev(dl), G.dev(dv)
                p = _lib.ptr
                for part in (_lib.BWD_TAIL, _lib.BWD_HEAD):
                    _lib.check(net._lib.paacb_backward_part(net.ctx, p(net.params), p(fwd['states']), b, p(fwd['ws']), p(dl_d),
                                                            p(dv_d), p(bws), p(grads), part, G.stream()), 'paacb_backward_part')
                torch.cuda.synchronize()
                assert_close(grads.cpu().numpy(), flat, 1e-5, 'TAIL + HEAD vs paacb_backward at r=8', elem_max=None)
    for bad in (-1, S):
        assert net._lib.paacb_set_sm_reserve(net.ctx, bad) == PAACB_EINVAL
