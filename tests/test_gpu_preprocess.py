"""GPU: paacb_preprocess_u8 against the oracle and the reference-generated golden sequence.  Bit-exact."""
import os

import numpy as np
import pytest
import torch

from oracle import preprocess as opre
from oracle.make_golden import gen_frames
from paac_b200.resize_tables import ROW, COL
import gpu_util as G

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def net():
    return G.make_net('NIPS', 4)


def test_golden_sequence_with_resets(net, golden_dir):
    g = np.load(os.path.join(golden_dir, 'preprocess_golden.npz'))
    n_envs, steps = int(g['n_envs']), int(g['steps'])
    frames = gen_frames(int(g['seed']), n_envs, int(g['n_pairs']))
    prev = np.zeros((n_envs, 84, 84, 4), np.uint8)
    for t in range(steps + 1):
        slots = np.zeros((n_envs, 4, 2, 210, 160), np.uint8)
        for e in range(n_envs):
            for j in range(4 if g['resets'][t, e] else 1):
                slots[e, j] = frames[e, g['used'][t, e, j]]
        nxt = G.preprocess(net, slots, 4, g['resets'][t], prev).cpu().numpy()
        assert (nxt == g['states'][t]).all(), 'step %d: %d bytes differ' % (t, (nxt != g['states'][t]).sum())
        prev = nxt


@pytest.mark.parametrize('n', [1, 2, 37, 300])
def test_random_vs_oracle(net, n):
    rng = np.random.RandomState(n)
    frames = rng.randint(0, 256, (n, 4, 2, 210, 160)).astype(np.uint8)
    prev = rng.randint(0, 256, (n, 84, 84, 4)).astype(np.uint8)
    reset = (rng.random_sample(n) < 0.3).astype(np.uint8)
    want = opre.step_states(prev, frames, reset, ROW, COL)
    got = G.preprocess(net, frames, 4, reset, prev).cpu().numpy()
    assert (got == want).all(), '%d bytes differ' % (got != want).sum()
    # single-slot layout, no reset flags
    want1 = opre.step_states(prev, frames[:, :1], np.zeros(n, np.uint8), ROW, COL)
    got1 = G.preprocess(net, np.ascontiguousarray(frames[:, :1]), 1, None, prev).cpu().numpy()
    assert (got1 == want1).all()


def test_in_place_and_empty(net):
    rng = np.random.RandomState(5)
    n = 9
    frames = rng.randint(0, 256, (n, 4, 2, 210, 160)).astype(np.uint8)
    prev = rng.randint(0, 256, (n, 84, 84, 4)).astype(np.uint8)
    reset = np.zeros(n, np.uint8)
    want = opre.step_states(prev, frames, reset, ROW, COL)
    buf = G.dev(prev)
    from paac_b200 import _lib
    f, r = G.dev(frames), G.dev(reset)
    _lib.check(net._lib.paacb_preprocess_u8(net.ctx, _lib.ptr(f), 4, _lib.ptr(r), _lib.ptr(buf), _lib.ptr(buf), n, G.stream()))
    _lib.check(net._lib.paacb_preprocess_u8(net.ctx, _lib.ptr(f), 4, _lib.ptr(r), _lib.ptr(buf), _lib.ptr(buf), 0, G.stream()))
    torch.cuda.synchronize()
    assert (buf.cpu().numpy() == want).all()
    rc = net._lib.paacb_preprocess_u8(net.ctx, _lib.ptr(f), 3, _lib.ptr(r), _lib.ptr(buf), _lib.ptr(buf), n, G.stream())
    assert rc == -1 and b'pairs_per_env' in net._lib.paacb_last_error()


def test_large_batch_properties(net):
    """Full-size check without the CPU oracle: shift property + max/resize computed with torch ops on the GPU."""
    n = 4096
    gen = torch.Generator(device='cuda'); gen.manual_seed(3)
    frames = torch.randint(0, 256, (n, 1, 2, 210, 160), dtype=torch.uint8, device='cuda', generator=gen)
    prev = torch.randint(0, 256, (n, 84, 84, 4), dtype=torch.uint8, device='cuda', generator=gen)
    out = torch.empty_like(prev)
    from paac_b200 import _lib
    _lib.check(net._lib.paacb_preprocess_u8(net.ctx, _lib.ptr(frames), 1, None, _lib.ptr(prev), _lib.ptr(out), n, G.stream()))
    torch.cuda.synchronize()
    assert torch.equal(out[..., :3], prev[..., 1:])
    mx = torch.maximum(frames[:, 0, 0], frames[:, 0, 1])
    row = torch.as_tensor(ROW, device='cuda', dtype=torch.long); col = torch.as_tensor(COL, device='cuda', dtype=torch.long)
    assert torch.equal(out[..., 3], mx[:, row][:, :, col])


@pytest.mark.parametrize('n', [5, 120, 300])
def test_zero_copy_from_pinned_host_frames(net, n):
    """The runners' frame buffers live in pinned, mapped host memory (Runners.pin()); the kernel reads them in place
    (narrow grid-stride launch for 96 < n <= the SM count, the copy pipeline on 32 CTAs above it).  Same bytes as with
    device-resident frames."""
    from paac_b200 import _lib
    rng = np.random.RandomState(100 + n)
    frames = torch.from_numpy(rng.randint(0, 256, (n, 4, 2, 210, 160)).astype(np.uint8)).pin_memory()
    prev = rng.randint(0, 256, (n, 84, 84, 4)).astype(np.uint8)
    reset = (rng.random_sample(n) < 0.3).astype(np.uint8)
    want = opre.step_states(prev, frames.numpy(), reset, ROW, COL)
    p, r = G.dev(prev), G.dev(reset)
    out = torch.empty_like(p)
    _lib.check(net._lib.paacb_preprocess_u8(net.ctx, frames.data_ptr(), 4, _lib.ptr(r), _lib.ptr(p), _lib.ptr(out), n,
                                            G.stream()), 'paacb_preprocess_u8')
    torch.cuda.synchronize()
    assert np.array_equal(out.cpu().numpy(), want)


def test_copy_pipeline_equals_cta_per_env_kernel():
    """Device-resident frames go through the persistent copy pipeline (one CTA per SM, 4 stages) when the row table is the
    affine default; any other table takes the CTA-per-environment kernel at the same size.  Both against the oracle, with
    the table each was given.  1,500 environments = more than 148 x 4: every stage of the ring is refilled; 20 % of the
    environments reset from their four pairs (out of place), and the single-pair layout runs in place."""
    import ctypes as C
    from paac_b200 import _lib
    n = 1500
    gen = torch.Generator(device='cuda'); gen.manual_seed(11)
    frames = torch.randint(0, 256, (n, 4, 2, 210, 160), dtype=torch.uint8, device='cuda', generator=gen)
    prev = torch.randint(0, 256, (n, 84, 84, 4), dtype=torch.uint8, device='cuda', generator=gen)
    reset = (torch.rand((n,), device='cuda', generator=gen) < 0.2).to(torch.uint8)
    assert int(reset.sum()) > 100
    f1 = frames[:, 0].contiguous()            # single-pair layout of the same frames (pairs = 1, no resets)
    frames_h, f1_h, prev_h, reset_h = frames.cpu().numpy(), f1[:, None].cpu().numpy(), prev.cpu().numpy(), reset.cpu().numpy()
    row_cta = ROW.copy()
    row_cta[5] += 1                           # breaks row(2k + 1) = row(1) + 5k: not expressible by the row-parity tensor maps
    for name, row in (('pipeline', ROW), ('cta', row_cta)):
        net = G.make_net('NIPS', 4)
        r32, c32 = np.ascontiguousarray(row, np.int32), np.ascontiguousarray(COL, np.int32)
        _lib.check(net._lib.paacb_set_resize_tables(net.ctx, r32.ctypes.data_as(C.POINTER(C.c_int32)),
                                                    c32.ctypes.data_as(C.POINTER(C.c_int32))), 'paacb_set_resize_tables')
        o = torch.empty_like(prev)
        _lib.check(net._lib.paacb_preprocess_u8(net.ctx, _lib.ptr(frames), 4, _lib.ptr(reset), _lib.ptr(prev), _lib.ptr(o), n, G.stream()))
        b = prev.clone()
        _lib.check(net._lib.paacb_preprocess_u8(net.ctx, _lib.ptr(f1), 1, None, _lib.ptr(b), _lib.ptr(b), n, G.stream()))
        torch.cuda.synchronize()
        want = opre.step_states(prev_h, frames_h, reset_h, row, COL)
        assert np.array_equal(o.cpu().numpy(), want), name
        want1 = opre.step_states(prev_h, f1_h, np.zeros(n, np.uint8), row, COL)
        assert np.array_equal(b.cpu().numpy(), want1), name + ', one pair in place'
