"""BASELINE.json configs[4]: synthetic 16,384 envs/GPU microbench -- the preprocessing (K1), n-step returns + loss gradient
(K7 + K8) and global-norm clip + RMSProp (K10 + K11) kernels against the HBM roofline.

    python tools/microbench_cfg5.py [--envs 16384] [--iters 30] > gpurun_out/micro_cfg5.json

Every launch is timed on its own with a CUDA event pair on the launching stream; between launches a 512 MB buffer is
rewritten so that nothing the next launch reads is left in the 126 MB L2 (K1's inputs are larger than L2 anyway: three
1.1 GB frame buffers rotate).  `achieved` = SURVEY 8(d) contract bytes / median launch time; `moved` is what the kernel
really transfers.  Peak = MEASURED_PEAKS.json hbm_gbs.
"""
import argparse, ctypes as C, json, os, statistics, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
from paac_b200 import _lib
from paac_b200.policy_v_network import NaturePolicyVNetwork


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--envs', type=int, default=16384)
    ap.add_argument('--iters', type=int, default=30)
    args = ap.parse_args()
    N, T, A = args.envs, 5, 6
    B = N * T
    dev = torch.device('cuda', 0)
    peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json'))) if os.path.exists(os.path.join(ROOT, 'MEASURED_PEAKS.json')) else {'hbm_gbs': 6650.0}
    peak = peaks['hbm_gbs']
    conf = dict(name='local_learning', num_actions=A, clip_norm=3.0, clip_norm_type='global', device='/gpu:0',
                entropy_regularisation_strength=0.02, seed=3, math='bf16x3')
    net = NaturePolicyVNetwork(conf)
    lib, ctx, p = net._lib, net.ctx, _lib.ptr
    st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    gen = torch.Generator(device=dev); gen.manual_seed(3)
    flush = torch.empty((512 << 20,), dtype=torch.uint8, device=dev)

    def time_launches(fn, iters, do_flush=True):
        for _ in range(3):
            fn(0)
        evs = []
        torch.cuda.synchronize()
        for i in range(iters):                      # everything is queued back to back: the GPU never waits for the host,
            if do_flush:                            # so an event pair brackets device time only
                flush.fill_(i & 255)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); fn(i); e1.record()
            evs.append((e0, e1))
        torch.cuda.synchronize()
        ms = [a.elapsed_time(b) for a, b in evs]
        return statistics.median(ms), min(ms)

    rows = []

    def row(name, med, best, contract, moved, unit_note):
        rows.append({'kernel': name, 'median_us': med * 1e3, 'best_us': best * 1e3, 'contract_bytes': contract,
                     'achieved_gbs': contract / med / 1e6, 'frac': contract / med / 1e6 / peak,
                     'moved_bytes': moved, 'moved_gbs': moved / med / 1e6, 'moved_frac': moved / med / 1e6 / peak,
                     'note': unit_note})

    # ---- K1 ----
    frames = [torch.randint(0, 256, (N, 1, 2, 210, 160), dtype=torch.uint8, device=dev, generator=gen) for _ in range(3)]
    prev = torch.randint(0, 256, (N, 84, 84, 4), dtype=torch.uint8, device=dev, generator=gen)
    nxt = torch.empty_like(prev)
    def k1(i):
        _lib.check(lib.paacb_preprocess_u8(ctx, p(frames[i % 3]), 1, None, p(prev), p(nxt), N, st), 'k1')
    med, best = time_launches(k1, args.iters, do_flush=False)
    row('preprocess_u8 (K1)', med, best, 33936.0 * N, 83328.0 * N,
        '%d env-steps per launch; contract 33,936 B/env-step (84 rows x 160 B x 2 frames + 7,056 B new plane); the kernel '
        'also reads and rewrites the 28,224 B interleaved stack (83,328 B moved)' % N)
    del frames, prev, nxt

    # ---- K7 + K8 ----
    f = lambda *s: torch.rand(s, device=dev, generator=gen)
    rewards = (f(T, N) * 4 - 2); over = (f(T, N) < 0.01).float(); values = f(T, N); boot = f(N)
    actions = torch.randint(0, A, (B,), dtype=torch.int32, device=dev, generator=gen)
    pi = torch.softmax(f(B, A) * 3, dim=1).contiguous(); v = f(B)
    y = torch.empty(B, device=dev); adv = torch.empty(B, device=dev); dl = torch.empty((B, A), device=dev)
    dv = torch.empty(B, device=dev); loss = torch.zeros(1, device=dev)
    def k78(i):
        _lib.check(lib.paacb_returns_loss_grad(ctx, p(rewards), p(over), p(values), p(boot), p(actions), p(pi), p(v), T, N,
                                               C.c_double(0.99), C.c_float(0.02), p(y), p(adv), p(dl), p(dv), p(loss), st), 'k78')
    med, best = time_launches(k78, args.iters)
    cb = 4.0 * (2 * A + 6) * B + 4.0 * N
    row('returns_loss_grad (K7+K8)', med, best, cb, cb, '%d training samples per launch, 72 B/sample at A=6 (+4 B/env bootstrap); '
        'includes the 4-byte memset node of the loss accumulator' % B)

    # ---- K10 + K11 ----
    P = net.param_count
    ms_ = torch.ones(P, device=dev); mom = torch.zeros(P, device=dev); grads = torch.randn(P, device=dev, generator=gen) * 0.01
    norm = torch.zeros(1, device=dev)
    ws = torch.zeros((int(lib.paacb_optimizer_workspace_floats(ctx)),), device=dev)
    def k1011(i):
        _lib.check(lib.paacb_clip_rmsprop(ctx, p(net.params), p(ms_), p(mom), p(grads), C.c_float(1.0), C.c_float(1e-6),
                                          C.c_float(0.99), C.c_float(0.1), C.c_float(0.0), C.c_float(3.0), _lib.CLIP_GLOBAL,
                                          p(norm), p(ws), st), 'k1011')
    med, best = time_launches(k1011, args.iters)
    row('clip_rmsprop (K10+K11, + the refresh of the forward weight images)', med, best, 28.0 * P, 28.0 * P,
        '%d parameters per launch, 28 B/param; the timed call also re-derives the bf16 / int8 operand images of the '
        'weights (4 small kernels) because paacb_clip_rmsprop owns that refresh' % P)
    lib.paacb_set_math(ctx, _lib.MATH_FP32)       # the optimizer alone: no operand images in fp32 mode
    med, best = time_launches(k1011, args.iters)
    row('clip_rmsprop (K10+K11) alone', med, best, 28.0 * P, 28.0 * P, '%d parameters per launch, 28 B/param' % P)

    # calibration of the method: a plain device copy moving the optimizer's byte volume, timed the same way
    src = torch.empty((int(14.0 * P),), dtype=torch.uint8, device=dev); dst = torch.empty_like(src)
    med, best = time_launches(lambda i: dst.copy_(src), args.iters)
    row('calibration: torch copy of 14 B x P (28 B/param moved)', med, best, 28.0 * P, 28.0 * P, 'same event-pair method')
    src = torch.empty((int(cb / 2),), dtype=torch.uint8, device=dev); dst = torch.empty_like(src)
    med, best = time_launches(lambda i: dst.copy_(src), args.iters)
    row('calibration: torch copy moving the K7+K8 byte volume', med, best, cb, cb, 'same event-pair method')

    print(json.dumps({'workload': 'BASELINE.json configs[4]: synthetic %d envs/GPU microbench, t_max 5, 6 actions, Nature' % N,
                      'peak_gbs': peak, 'peak_source': 'MEASURED_PEAKS.json hbm_gbs (copy bandwidth)', 'iters': args.iters,
                      'timing': 'one CUDA event pair per launch, launches queued back to back, 512 MB L2 flush between launches (K1: inputs > L2)',
                      'rows': rows}, indent=1))


if __name__ == '__main__':
    main()
