#!/usr/bin/env python
"""bench.py -- PAAC env-steps/sec (Nature CNN, t_max=5) on N B200s; update ms.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--envs E] [--math fp32|tf32x3|tf32]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

A "step" is one PAAC update cycle of the hot path over one batch of synthetic input (BASELINE.json configs[2]:
synthetic raw 210x160 frames, NatureNetwork, 4096 envs per GPU, t_max = 5, 6 actions):
    5 x [ policy forward on 4096 states + categorical sampling, preprocessing of 4096 raw frame pairs ]
    + bootstrap forward, training forward on 20,480 states, n-step returns + loss gradient, backward,
    [NCCL allreduce of the flat gradient when N > 1], global-norm clip + RMSProp.
One step = 20,480 env-steps per GPU.  `value` = env-steps of all ranks / max-over-ranks device time with the
frames resident in HBM; `e2e` = the same cycle driven from HOST buffers (pinned frames uploaded and sampled
actions read back every env step, loss read back every update).  Rank 0 prints ONE JSON line.

--dump-outputs DIR: right after the K timed steps of the headline, rank 0 writes what the last of them computed as
DIR/<name>.npy (float32; see dump_outputs()).  The inputs are seeded, so two builds run with the same arguments can be
compared output for output.

--impl reference times the CPU restatement of the reference's path (oracle/cpu_baseline.py; TF1/ALE cannot be
installed here) on the host cores for the same metric/config, each step a bounded sample of the workload.
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = 'paac_env_steps_per_sec'
UNIT = 'env-steps/s'
T_MAX = 5
NUM_ACTIONS = 6
FRAME_PAIR_BYTES = 2 * 210 * 160
K1_ALGO_BYTES = 33936            # SURVEY 8d: 84 rows x 160 B x 2 frames read + 7,056 B written per env-step
K1_MOVED_BYTES = 26880 + 2 * 28224      # what the kernel moves: the selected rows + the interleaved stack read and rewritten


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=40)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--envs', type=int, default=4096, help='environments per GPU')
    ap.add_argument('--arch', default='NATURE', choices=['NATURE', 'NIPS'])
    ap.add_argument('--math', default=os.environ.get('PAACB_BENCH_MATH', 'auto'), choices=['auto', 'fp32', 'tf32x3', 'tf32', 'bf16x3'],
                    help="'auto': bf16x3 (the parity-grade tensor-core path, both architectures)")
    ap.add_argument('--frame_pool', type=int, default=8, help='device frame buffers rotated between env steps')
    ap.add_argument('--no_cpu_baseline', action='store_true')
    ap.add_argument('--no_e2e', action='store_true')
    ap.add_argument('--no_variants', action='store_true')
    ap.add_argument('--no_overlap_allreduce', action='store_true', help='N > 1: one all-reduce after the whole backward')
    ap.add_argument('--e2e_slices', type=int, default=2, help='environment slices pipelined in the end-to-end arm')
    ap.add_argument('--dev_slices', type=int, default=1,
                    help='device-resident arm: contiguous environment slices, each rolled out on its own stream (1 = whole batch on one stream)')
    ap.add_argument('--ref_envs', type=int, default=64, help='--impl reference: envs per step (bounded sample)')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write what the last timed step computed to DIR/<name>.npy (float32, under 64 MB in all)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs writes the outputs of the B200 arm')
    if args.math == 'auto':
        args.math = 'bf16x3'
    return args


def workload_config(args, n_gpus):
    return {'workload': 'BASELINE.json configs[2]: synthetic raw 210x160 uint8 frame pairs, %sNetwork, %d envs/GPU, '
                        't_max=%d, %d actions, learner-only (frames resident in HBM)' % (
                            'Nature' if args.arch == 'NATURE' else 'NIPS', args.envs, T_MAX, NUM_ACTIONS),
            'arch': args.arch, 'envs_per_gpu': args.envs, 't_max': T_MAX, 'num_actions': NUM_ACTIONS,
            'env_steps_per_step': args.envs * T_MAX * n_gpus,
            'rollout_schedule': ('whole batch on one stream' if args.dev_slices <= 1 else
                                 '%d contiguous environment slices, one stream each (act -> observe per slice in order; one update '
                                 'on the whole batch)' % args.dev_slices),
            'parallelism': 'envs sharded over %d GPU(s); flat fp32 gradient all-reduced per update (NCCL; the fc + heads tail '
                           'under the conv weight-gradient kernels, the conv head after them)' % n_gpus,
            'l2': 'inputs larger than L2: each env step reads a different %d-deep rotating frame buffer of %.0f MB and '
                  'the update streams %.2f GB of activations (L2 = 126 MB)' % (
                      args.frame_pool, args.envs * FRAME_PAIR_BYTES / 1e6, args.envs * T_MAX * 21632 * 4 * 2 / 1e9)}


# ---------------------------------------------------------------------------------------------------------
# reference arm: the CPU restatement on the host cores
# ---------------------------------------------------------------------------------------------------------
def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    from oracle import cpu_baseline
    cores = os.cpu_count() or 1
    warm = max(args.warmup, 3)              # the same warm-up rule as the B200 arm
    sps, ms, done, cores = cpu_baseline.time_cycles(args.arch, args.ref_envs, T_MAX, NUM_ACTIONS, steps=args.steps,
                                                    warmup=warm, cores=cores, max_seconds=240)
    sample = ('restated reference CPU path (oracle port, not TF1): %d timed update cycles (after %d warm-up cycles) of %d envs x '
              't_max %d -- a bounded sample of the %d-env workload: the CPU rate per env-step does not depend on the env count '
              'beyond this size -- torch-CPU fp32 + NumPy preprocessing, %d threads' % (done, warm, args.ref_envs, T_MAX, args.envs, cores))
    cfg = workload_config(args, 1)
    # what this arm really ran: the bounded sample, on the host cores of ONE process whatever --gpus says
    cfg.update(envs_timed=args.ref_envs, env_steps_per_step=args.ref_envs * T_MAX,
               workload=cfg['workload'] + ' [reference arm: %d-env bounded sample per step on %d host threads]' % (args.ref_envs, cores),
               parallelism='host CPU only (rank 0); at --gpus N > 1 this is still ONE CPU run, not N')
    line = {'impl': 'reference', 'metric': METRIC, 'value': sps, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': done,
            'warmup': warm, 'ms_per_step': ms, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic', 'config': cfg,
            'cpu_baseline': {'value': sps, 'unit': UNIT, 'cores': cores, 'kind': 'port', 'sample': sample},
            'e2e': {'value': sps, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'gpu_launches': 0}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------------------
class ClockSampler(object):
    """SM clock / throttle reasons / power sampled DURING the timed region by an NVML thread (every ~5 ms; NVML calls drop the
    GIL).  Falls back to an `nvidia-smi -lms` child when pynvml is missing."""
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        import threading
        self.rows, self.p, self.f, self.th = [], None, None, None
        self.stop_flag = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            visible = os.environ.get('CUDA_VISIBLE_DEVICES')
            phys = int(visible.split(',')[index]) if visible and visible.split(',')[index].isdigit() else index
            h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            bits = {'hw_slowdown': pynvml.nvmlClocksThrottleReasonHwSlowdown,
                    'hw_thermal_slowdown': pynvml.nvmlClocksThrottleReasonHwThermalSlowdown,
                    'sw_thermal_slowdown': pynvml.nvmlClocksThrottleReasonSwThermalSlowdown,
                    'sw_power_cap': pynvml.nvmlClocksThrottleReasonSwPowerCap}

            def loop():
                while not self.stop_flag.is_set():
                    try:
                        mhz = float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                        mask = int(pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h))
                        watts = pynvml.nvmlDeviceGetPowerUsage(h) / 1e3
                        self.rows.append((mhz, watts, [n for n, b in bits.items() if mask & b]))
                    except Exception:
                        pass
                    time.sleep(0.005)
            self.th = threading.Thread(target=loop, daemon=True)
            self.th.start()
            return
        except Exception:
            self.th = None
        self.f = tempfile.NamedTemporaryFile('w+', suffix='.csv', delete=False)
        try:
            self.p = subprocess.Popen(['nvidia-smi', '-i', str(index), '--query-gpu=' + self.Q,
                                       '--format=csv,noheader,nounits', '-lms', '20'], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': [], 'samples': 0}
        if self.th is not None:
            self.stop_flag.set()
            self.th.join(1.0)
            if self.rows:
                reasons = set()
                for r in self.rows:
                    reasons.update(r[2])
                out.update(sm_mhz=statistics.median(r[0] for r in self.rows), sm_max_mhz=self.max_mhz,
                           reasons=sorted(reasons), samples=len(self.rows), power_w_max=max(r[1] for r in self.rows),
                           source='nvml thread, 5 ms period, timed region only')
            return out
        if self.p is None:
            return out
        time.sleep(0.05)
        self.p.terminate()
        try:
            self.p.wait(5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(', ') for r in open(self.f.name) if r.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons, pw = [], [], set(), []
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for r in rows:
            if len(r) < 8:
                continue
            try:
                sm.append(float(r[0])); mx.append(float(r[1])); pw.append(float(r[2]))
            except ValueError:
                continue
            for nm, val in zip(names, r[4:8]):
                if val.strip().lower() == 'active':
                    reasons.add(nm)
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm),
                       power_w_max=max(pw), source='nvidia-smi -lms 20')
        return out


# ---------------------------------------------------------------------------------------------------------
# the B200 arm
# ---------------------------------------------------------------------------------------------------------
def load_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return d['hbm_gbs'], d['bf16_tflops'], d.get('bf16_tflops_sustained', d['bf16_tflops']), 'measured'
    return 6650.0, 1590.0, 1400.0, 'fallback'


def load_umma_peaks():
    """tools/probe/umma_peak on a B200 (profiles/r02_umma_peaks.json): what ONE CTA per SM issues per tcgen05.mma kind and N."""
    try:
        return json.load(open(os.path.join(ROOT, 'profiles', 'r02_umma_peaks.json')))['peaks']
    except Exception:
        return None


def layer_macs(arch):
    """MACs per sample of each conv/fc layer: (name, macs, has_dgrad)."""
    if arch == 'NATURE':
        return [('conv1', 400 * 256 * 32, False), ('conv2', 81 * 512 * 64, True), ('conv3', 49 * 576 * 64, True),
                ('fc4', 3136 * 512, True)]
    return [('conv1', 400 * 256 * 16, False), ('conv2', 81 * 256 * 32, True), ('fc3', 2592 * 256, True)]


def layer_bytes(arch, kind, li, elem_in, state_bytes=28224):
    """Compulsory HBM bytes per sample of one conv/fc kernel: operands read once + result written once, at the storage
    widths of the arithmetic mode (activations / dZ: 4 bytes per element in every mode -- fp32, or two bf16 planes; the
    uint8 state: 1 byte; the ReLU-mask plane a data-gradient kernel reads: 2 bytes per element in bf16x3, 4 otherwise)."""
    if arch == 'NATURE':
        elems = [20 * 20 * 32, 9 * 9 * 64, 7 * 7 * 64, 512]
    else:
        elems = [20 * 20 * 16, 9 * 9 * 32, 256]
    x_in = state_bytes if li == 0 else 4 * elems[li - 1]
    y_out = 4 * elems[li]
    if kind in ('fwd', 'wgrad'):
        return x_in + y_out                       # fwd: read X, write Y; wgrad: read X and dZ (the small dW is atomics in L2)
    return y_out + elem_in * elems[li - 1] + 4 * elems[li - 1]      # dgrad: read dZ + mask plane of X, write dX


def read_profile(net):
    lib = net._lib
    out = {}
    for s in range(lib.paacb_profile_slots()):
        name = C.create_string_buffer(64)
        ms, cnt = C.c_double(), C.c_int64()
        lib.paacb_profile_read(net.ctx, s, name, 64, C.byref(ms), C.byref(cnt))
        if cnt.value > 0:
            out[name.value.decode()] = (ms.value, cnt.value)
    return out


def bind_to_gpu_numa_node(local):
    """Run this rank on the CPUs that are local to its GPU, BEFORE the pinned frame buffers are allocated: the kernel reads
    them over PCIe, and first-touch puts the pages on the node of the allocating thread.  Without it two ranks on one host
    halved each other's end-to-end rate (remote-socket reads).  Best effort: silently skipped where NVML says nothing."""
    try:
        import pynvml
        pynvml.nvmlInit()
        visible = os.environ.get('CUDA_VISIBLE_DEVICES')
        index = int(visible.split(',')[local]) if visible and visible.split(',')[local].isdigit() else local
        handle = pynvml.nvmlDeviceGetHandleByIndex(index)
        ncpu = os.cpu_count() or 1
        mask = pynvml.nvmlDeviceGetCpuAffinity(handle, (ncpu + 63) // 64)
        allowed = os.sched_getaffinity(0)
        cpus = [i for i in range(ncpu) if ((mask[i // 64] >> (i % 64)) & 1) and i in allowed]
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return 0


DUMP_ENVS = 4096            # --dump-outputs: per-environment outputs of at most this many environments (a seeded sample)
DUMP_STATE_ENVS = 16        # and the preprocessed observations (28,224 B per environment and env step) of this many


def dump_outputs(eng, out_dir):
    """Write what the last update cycle of `eng` hands its caller to out_dir/<name>.npy as float32 (per-step arrays as
    [T, n, ...]).  The n environments are a fixed seeded sample (env_index.npy), so the files stay under 64 MB at any --envs:
    about 1.5 MB of per-environment outputs, 9 MB of observations and 20 MB of parameters, gradient and RMSProp slot
    (Nature, 6 actions)."""
    import numpy as np
    import torch
    T, N = eng.T, eng.N
    pick = np.sort(np.random.RandomState(0).choice(N, min(N, DUMP_ENVS), replace=False))
    spick = pick[np.sort(np.random.RandomState(1).choice(len(pick), min(len(pick), DUMP_STATE_ENVS), replace=False))]
    idx, sidx = torch.from_numpy(pick).to(eng.dev), torch.from_numpy(spick).to(eng.dev)
    per_step = lambda x: x.reshape((T, N) + x.shape[1:])[:, idx]
    # the T observations of the rollout just trained on: s_1 .. s_{T-1} in the half update() rolled away from, s_T in slot 0
    # of the current half
    observed = torch.cat([eng._sbuf[1 - eng._cur, 1:], eng.state(0)[None]])[:, sidx]
    out = {'env_index': idx, 'observed_states': observed,
           'actions': eng.actions[:, idx], 'values': eng.values[:, idx], 'bootstrap_values': eng.boot_v[idx],
           'pi': per_step(eng.pi), 'v': per_step(eng.v), 'returns': per_step(eng.y), 'advantages': per_step(eng.adv),
           'dlogits': per_step(eng.dlogits), 'dv': per_step(eng.dv),
           'loss': eng.loss, 'global_norm': eng.norm, 'grads': eng.grads, 'params': eng.net.params, 'rmsprop_ms': eng.ms}
    os.makedirs(out_dir, exist_ok=True)
    total = 0
    for name, t in out.items():
        a = t.detach().float().cpu().numpy()
        np.save(os.path.join(out_dir, name + '.npy'), a)
        total += a.nbytes
    return {'dir': out_dir, 'arrays': len(out), 'bytes': total, 'envs_sampled': len(pick), 'state_envs_sampled': len(sidx)}


def run_b200(args):
    import numpy as np
    import torch
    from paac_b200 import _lib
    from paac_b200.engine import RolloutEngine
    from paac_b200.policy_v_network import NaturePolicyVNetwork, NIPSPolicyVNetwork

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise SystemExit('bench.py: no CUDA device; the B200 arm has no CPU fallback (use --impl reference)')
    all_cpus = os.sched_getaffinity(0)
    numa_cpus = bind_to_gpu_numa_node(local)
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        torch.distributed.init_process_group('nccl', device_id=dev)
    N, T, A = args.envs, T_MAX, NUM_ACTIONS
    conf = dict(name='local_learning', num_actions=A, clip_norm=3.0, clip_norm_type='global', device='/gpu:%d' % local,
                entropy_regularisation_strength=0.02, seed=3, math=args.math)
    net = (NaturePolicyVNetwork if args.arch == 'NATURE' else NIPSPolicyVNetwork)(conf)
    eng = RolloutEngine(net, N, T, seed=3 * (rank + 1), world_size=world, overlap_allreduce=not args.no_overlap_allreduce)
    P = net.param_count

    gen = torch.Generator(device=dev)
    gen.manual_seed(3 * (rank + 1))                                  # mirrors atari_emulator.py:18
    pool = [torch.randint(0, 256, (N, 1, 2, 210, 160), dtype=torch.uint8, device=dev, generator=gen)
            for _ in range(args.frame_pool)]
    u = torch.rand((T, N), device=dev, generator=gen)
    rewards = torch.where(u < 0.05, -1.0, torch.where(u > 0.95, 1.0, 0.0)).float()
    over = (torch.rand((T, N), device=dev, generator=gen) < 0.01).float()
    eng.state(0).copy_(torch.randint(0, 256, eng.state(0).shape, dtype=torch.uint8, device=dev, generator=gen))
    lr = 0.0224
    counter = [0]

    def step_device():
        for t in range(T):
            eng.act(t)
            buf = pool[counter[0] % len(pool)]
            counter[0] += 1
            eng.observe_frames(t, buf.data_ptr(), 1, None, rewards[t], over[t])
        eng.update(lr)

    def make_step_sliced(S):
        # The rollout as S contiguous environment slices (what the runners' workers own, runners.py:17-18), each on its own
        # stream: every environment still sees act -> step -> observe in order and the update is the whole batch, so the
        # results are the same bits (tests/test_gpu_engine.py: sliced == whole-batch); the kernels of one slice fill the
        # SMs the other slice's kernels leave idle while they start up and drain.
        bounds = [(c * N // S, (c + 1) * N // S) for c in range(S)]
        streams = [torch.cuda.Stream(dev) for _ in bounds]
        ev_done = [torch.cuda.Event() for _ in bounds]
        ev_upd = torch.cuda.Event()

        def step():
            main = torch.cuda.current_stream(dev)
            ev_upd.record(main)
            for c, (lo, hi) in enumerate(bounds):
                streams[c].wait_event(ev_upd)
                with torch.cuda.stream(streams[c]):
                    for t in range(T):
                        eng.act(t, lo, hi)
                        buf = pool[(counter[0] + t) % len(pool)]
                        eng.observe_frames(t, buf.data_ptr() + lo * FRAME_PAIR_BYTES, 1, None, rewards[t], over[t], lo, hi)
                    eng.bootstrap(lo, hi)
                    ev_done[c].record(streams[c])
            counter[0] += T
            for e in ev_done:
                main.wait_event(e)
            eng.update(lr)
        return step

    if args.dev_slices > 1:
        step_device = make_step_sliced(min(args.dev_slices, N))

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize(dev)

    def timed(fn, k):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(k):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            torch.distributed.all_reduce(ms, op=torch.distributed.ReduceOp.MAX)
        return float(ms.item())

    # ---- device-resident arm ---------------------------------------------------------------------------
    for _ in range(max(args.warmup, 3)):
        step_device()
    barrier()
    # pass 1 -- the headline: K steps, nothing but the hot path on the stream
    launches0 = net.launch_count()
    clocks = ClockSampler(local)
    ms_plain = timed(step_device, args.steps)
    clk = clocks.stop()
    launches = net.launch_count() - launches0
    dumped = dump_outputs(eng, args.dump_outputs) if args.dump_outputs and rank == 0 else None
    ms_per_step = ms_plain / args.steps
    value = world * N * T * args.steps / (ms_plain / 1e3)
    # pass 2 -- the same K steps with every kernel bracketed by a CUDA event pair on the launching stream (the per-kernel
    # roofline table); the event records cost ~1 % of the step, which is why the headline is not taken from this pass
    _lib.check(net._lib.paacb_profile_enable(net.ctx, 1))
    _lib.check(net._lib.paacb_profile_reset(net.ctx))
    ms_total = timed(step_device, args.steps)
    prof = read_profile(net)
    _lib.check(net._lib.paacb_profile_enable(net.ctx, 0))
    loss_val = float(eng.loss.item())

    # ---- per-kernel roofline table (device time from CUDA events on the launching stream) ---------------
    hbm_peak, tc_burst, tc_sust, peak_kind = load_peaks()
    # SURVEY 8(d): conv / FC kernels are held against the TENSOR roofline -- algorithmic flops (2 x MACs of the layer, whatever
    # the number of MMAs the split arithmetic issues) / device time / peak -- with the HBM fraction of the same kernel beside
    # it.  Kernels are timed inside a long step -> the sustained figure of MEASURED_PEAKS.json (a cuBLAS bf16 GEMM).  The
    # other tcgen05 kinds scale it by the ratio tools/probe/umma_peak measured on this pool (kind::tf32 / kind::i8 vs
    # kind::f16 at N = 256); without that file: tf32 = 1/2, i8 = 2 (the architectural ratios).
    bf16_math = args.math == 'bf16x3'
    up = load_umma_peaks()
    r_tf32 = (up['tf32']['N256'] / up['f16_bf16']['N256']) if up else 0.5
    r_i8 = (up['i8']['N256'] / up['f16_bf16']['N256']) if up else 2.0
    tf32_peak = tc_sust if bf16_math else r_tf32 * tc_sust
    i8_peak = r_i8 * tc_sust
    peak_note = ('bf16_tflops_sustained (kind::f16 on bf16-split operands, 3 MMAs per algorithmic product: 1/3 is the ceiling)'
                 if bf16_math else
                 '%.2f x bf16_tflops_sustained (kind::tf32; ratio %s)' % (r_tf32, 'measured, profiles/r02_umma_peaks.json' if up else 'architectural'))
    B = N * T
    fwd_samples = (T * N + N + B) * args.steps       # acting + bootstrap + training forward
    kernels = []
    for li, (lname, macs, has_dgrad) in enumerate(layer_macs(args.arch)):
        for kind, samples in (('fwd', fwd_samples), ('wgrad', B * args.steps), ('dgrad', B * args.steps if has_dgrad else 0)):
            key = '%s_%s' % (lname, kind)
            if key in prof and samples:
                ms, cnt = prof[key]
                ach = 2.0 * macs * samples / (ms / 1e3) / 1e12
                nbytes = float(layer_bytes(args.arch, kind, li, 2 if bf16_math else 4)) * samples
                ach_b = nbytes / (ms / 1e3) / 1e9
                # conv1 forward runs on the int8 pipe in every tensor-core mode (tc2_conv1.cu)
                i8 = (li == 0 and kind == 'fwd' and args.math != 'fp32')
                peak = i8_peak if i8 else tf32_peak
                row = {'name': key, 'ms': ms, 'launches': cnt, 'frac_tensor': ach / peak, 'tflops': ach,
                       'frac_hbm': ach_b / hbm_peak, 'gbs': ach_b, 'hbm_bytes_per_launch': nbytes / cnt,
                       'bound': 'tensor', 'achieved': ach, 'peak': peak, 'unit': 'TFLOP/s', 'frac': ach / peak,
                       'algo_per_launch': 2.0 * macs * samples / cnt,
                       'peak_note': ('%.2f x bf16_tflops_sustained (kind::i8)' % r_i8) if i8 else peak_note}
                kernels.append(row)
    def hbm_row(key, bytes_total):
        if key in prof:
            ms, cnt = prof[key]
            ach = bytes_total / (ms / 1e3) / 1e9
            kernels.append({'name': key, 'ms': ms, 'launches': cnt, 'bound': 'hbm', 'achieved': ach, 'peak': hbm_peak,
                            'unit': 'GB/s', 'frac': ach / hbm_peak, 'algo_per_launch': bytes_total / cnt})
    hbm_row('preprocess_u8', float(K1_ALGO_BYTES) * N * T * args.steps)
    for k in kernels:
        if k['name'] == 'preprocess_u8':
            # the contract counts the new plane only; the kernel also reads and rewrites the 28,224 B interleaved stack that
            # conv1's operand layout needs (DESIGN 3): report what it really moves beside the contract figure
            moved = float(K1_MOVED_BYTES) * N * T * args.steps
            k['moved_gbs'] = moved / (k['ms'] / 1e3) / 1e9
            k['moved_frac'] = k['moved_gbs'] / hbm_peak
    hbm_row('returns_loss_grad', (4.0 * (2 * A + 6) * B + 4.0 * N) * args.steps)
    hbm_row('grad_sumsq', 4.0 * P * args.steps)
    # fused cooperative optimizer: one kernel carries the whole K10 + K11 contract (28 B/param); two-launch version: 4 + 24
    hbm_row('clip_rmsprop', (24.0 if 'grad_sumsq' in prof else 28.0) * P * args.steps)
    F = 512 if args.arch == 'NATURE' else 256
    hbm_row('heads_fwd', 4.0 * F * (T * N + N + B) * args.steps)       # reads the hidden activations once
    hbm_row('heads_bwd', 8.0 * F * B * args.steps)                     # reads h, writes dh
    # measured DRAM traffic (dram__bytes_read + write from `ncu --set full`, tools/ncu_dram_table.py) per unit, committed
    # under profiles/: traffic per launch = bytes per sample x the samples an average launch of that kernel processes
    dram_table, dram_src = {}, None
    try:
        for name in ('r02_ncu_dram_bytes.json', 'r01_ncu_dram_bytes.json'):
            path = os.path.join(ROOT, 'profiles', name)
            if os.path.exists(path):
                dj = json.load(open(path))
                if dj.get('arch', 'NATURE') == args.arch:
                    dram_table, dram_src = dj['kernels'], dj['source']
                    break
    except Exception:
        pass
    units_total = {'preprocess_u8': N * T * args.steps, 'heads_fwd': fwd_samples, 'heads_bwd': B * args.steps}
    for k in kernels:
        kind = k['name'].rsplit('_', 1)[-1]
        units = units_total.get(k['name'], fwd_samples if kind == 'fwd' else B * args.steps)
        if bf16_math and k['name'] in dram_table:
            dt = dram_table[k['name']]
            k['traffic'] = dt['dram_bytes_per_unit'] * units / k['launches']
            # what ncu saw for ONE launch of this kernel at the captured batch (cold, serialised): DRAM rate against the same
            # HBM peak and tensor-pipe activity -- which of the two roofs the kernel is really near (DESIGN 3.3)
            cap_units = dj.get('envs' if k['name'] == 'preprocess_u8' else 'batch')
            if cap_units and dt.get('duration_us'):
                k['ncu_dram_frac'] = dt['dram_bytes_per_unit'] * cap_units / (dt['duration_us'] * 1e-6) / 1e9 / hbm_peak
                k['ncu_tensor_pipe_active'] = dt.get('tensor_pipe_active_pct', 0.0) / 100.0
    accounted = sum(k['ms'] for k in kernels)
    for k in kernels:
        k['share_of_step'] = k['ms'] / ms_total
    kernels.sort(key=lambda k: -k['ms'])
    dom = kernels[0]
    roofline = {'kernel': dom['name'], 'bound': dom['bound'], 'achieved': dom['achieved'], 'peak': dom['peak'],
                'unit': dom['unit'], 'frac': dom['frac'], 'traffic': dom.get('traffic'), 'traffic_source': dram_src,
                'share_of_step': dom['share_of_step'],
                'launches': dom['launches'], 'avg_launch_ms': dom['ms'] / dom['launches'],
                'algo_per_launch': dom['algo_per_launch'],
                'frac_tensor': dom.get('frac_tensor'), 'frac_hbm': dom.get('frac_hbm'),
                'peak_source': ('%s: MEASURED_PEAKS.json ' % peak_kind) +
                               (dom.get('peak_note', peak_note) if dom['bound'] == 'tensor' else 'hbm_gbs (copy bandwidth)'),
                'rule': 'SURVEY 8(d): conv / FC kernels against the tensor roofline in ALGORITHMIC flops (frac_hbm beside it), '
                        'K1 / heads / returns / optimizer against HBM; dominant kernel = largest share of the profiled step',
                'tcgen05_peaks_one_cta_per_sm': up}
    # nominal whole-step fraction: contract flops per env-step / tf32 peak
    flops_per_env_step = 71.96e6 if args.arch == 'NATURE' else 21.65e6
    step_frac = (value / world) * flops_per_env_step / 1e12 / tf32_peak

    # ---- variant: the acting forwards write the training workspace, update() runs no second forward -----------
    # (same bits, tests/test_gpu_tc.py::test_training_forward_schedules_are_bit_identical).  Reported beside the headline,
    # never as it: `value` above keeps the reference's schedule with the full training forward inside the timed region.
    variants = {}
    if not args.no_variants:
        eng.set_train_forward('reuse')
        for _ in range(3):
            step_device()
        r_ms = timed(step_device, args.steps)
        variants['reuse_acting_activations'] = {
            'value': world * N * T * args.steps / (r_ms / 1e3), 'unit': UNIT, 'ms_per_step': r_ms / args.steps,
            'note': "RolloutEngine(train_forward='reuse'): act(t) stores its activations in the training workspace "
                    '(paacb_policy_forward_at) and the update skips the redundant training forward; bit-identical results'}
        eng.set_train_forward('batched')
        # the reference's DEFAULT size (train.py:95-96, BASELINE.json configs[0], [1], [3]: 32 environments per GPU): one cycle
        # is ~60 small launches, so the engine replays act / update as CUDA graphs (tools/small_batch.py has the full table)
        if rank == 0 and world == 1:
            try:
                import importlib.util
                spec = importlib.util.spec_from_file_location('small_batch', os.path.join(ROOT, 'tools', 'small_batch.py'))
                sb = importlib.util.module_from_spec(spec)
                spec.loader.exec_module(sb)
                r32 = sb.engine_numbers(args.arch, 32, 100, True, math=args.math)
                variants['envs_32_graph_replay'] = {
                    'value': r32['env_steps_per_s'], 'unit': UNIT, 'ms_per_step': r32['ms_per_cycle'], 'update_ms': r32['update_ms'],
                    'note': '32 environments x t_max 5 on one GPU (the reference default -ec 32), act / update replayed as CUDA '
                            'graphs, device-resident raw frames; %d kernel launches issued per cycle' % r32['kernel_launches_issued_per_cycle']}
            except Exception as e:                      # a variant, never the headline: report and go on
                variants['envs_32_graph_replay'] = {'error': str(e)[:200]}

    # ---- end-to-end arm: host buffers in, actions / loss out ---------------------------------------------
    e2e = None
    if not args.no_e2e:
        # The runners' raw frames live in pinned, mapped host memory (paac_b200/runners.py: Runners.pin()); the
        # preprocessing kernel reads the 84 + 84 source rows it needs STRAIGHT from there over PCIe (zero-copy, UVA):
        # 26,880 of the 67,200 bytes of a frame pair cross the bus, and there is no staging copy in HBM.
        host_frames = [torch.randint(0, 256, (N, 1, 2, 210, 160), dtype=torch.uint8).pin_memory() for _ in range(2)]
        host_rew, host_over = rewards.cpu().pin_memory(), over.cpu().pin_memory()
        host_onehot = torch.empty((N, A), dtype=torch.float32).pin_memory()
        host_loss = torch.empty((1,), dtype=torch.float32).pin_memory()
        stream = torch.cuda.current_stream(dev)
        io_stream = torch.cuda.Stream(dev)
        tf_stream = torch.cuda.Stream(dev)
        ev_tf = torch.cuda.Event()
        # the FULL training forward runs, but step by step on a side stream while the frames of the next env step cross
        # PCIe (the SMs are otherwise idle then) instead of in one piece inside update(): same work, same bits
        eng.set_train_forward('stepwise')
        S = max(1, min(args.e2e_slices, N))
        bounds = [(c * N // S, (c + 1) * N // S) for c in range(S)]       # contiguous env slices, like the runners' workers
        ev_act = [torch.cuda.Event() for _ in bounds]
        ev_obs = [torch.cuda.Event() for _ in bounds]

        def step_host():
            # Lock-step PAAC with the environment slices pipelined: slice c's actions go back to the host as soon as its
            # forward is done, its environments step (here: the pre-generated frames), and its frame ingestion (PCIe-bound)
            # overlaps the next slice's forward.  Every slice still sees act -> step -> observe in order: same results.
            for t in range(T):
                for c, (lo, hi) in enumerate(bounds):
                    if t > 0:
                        stream.wait_event(ev_obs[c])                          # states[t] of this slice are complete
                    # the heads kernel writes the one-hot actions straight into pinned, mapped host memory (what the
                    # runners' shared action array is): the environments need the actions, nothing else comes back
                    eng.act(t, lo, hi, onehot_out=host_onehot[lo:hi])
                    ev_act[c].record(stream)
                tf_stream.wait_event(ev_act[S - 1])                           # states[t] complete (every slice's act waited for it)
                with torch.cuda.stream(tf_stream):
                    eng.train_forward_step(t)
                for c, (lo, hi) in enumerate(bounds):
                    ev_act[c].synchronize()                                   # host has this slice's actions: its envs step
                    with torch.cuda.stream(io_stream):
                        # the raw frames are read by the kernel from pinned host memory inside the timed region
                        eng.observe_frames(t, host_frames[t & 1].data_ptr() + lo * FRAME_PAIR_BYTES, 1, None, host_rew[t],
                                           host_over[t], lo, hi)
                        ev_obs[c].record(io_stream)
            for c, (lo, hi) in enumerate(bounds):
                stream.wait_event(ev_obs[c])
                eng.bootstrap(lo, hi)                                         # V(s_T) of this slice under the next slice's frames
            ev_tf.record(tf_stream)
            stream.wait_event(ev_tf)
            eng.update(lr)
            host_loss.copy_(eng.loss, non_blocking=True)
            stream.synchronize()

        for _ in range(2):
            step_host()
        e_steps = max(2, args.steps // 2)
        e_ms = timed(step_host, e_steps)
        eng.set_train_forward('batched')
        e2e = {'value': world * N * T * e_steps / (e_ms / 1e3), 'unit': UNIT, 'steps': e_steps,
               'ms_per_step': e_ms / e_steps,
               'h2d_bytes_per_step': T * (N * 2 * 84 * 160 + 2 * 4 * N), 'd2h_bytes_per_step': T * N * A * 4 + 4,
               'host_bytes_per_step': T * N * FRAME_PAIR_BYTES, 'env_slices': S, 'cpus_bound_to_gpu_node': numa_cpus,
               'train_forward': 'stepwise (full training forward, issued per env step on a side stream under the PCIe reads)',
               'api': 'RolloutEngine.act / observe_frames / update over the C ABI; every env step the raw 210x160 frame '
                      'pairs are read by paacb_preprocess_u8 directly from pinned mapped host memory (zero-copy: the 84 '
                      'selected rows of both frames cross PCIe = h2d_bytes_per_step) and the sampled one-hot actions are '
                      'read back; the loss is read back every update'}

    # ---- CPU baseline beside it (rank 0, N = 1 only; bounded sample) ---------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        os.sched_setaffinity(0, all_cpus)               # the CPU baseline gets every host core again
        from oracle import cpu_baseline
        c_envs = 32
        sps, cms, done, cores = cpu_baseline.time_cycles(args.arch, c_envs, T, A, steps=1000, warmup=1, max_seconds=15)
        cpu = {'value': sps, 'unit': UNIT, 'cores': cores, 'kind': 'port',
               'sample': 'restated reference CPU path (oracle port, not TF1): %d update cycles of %d envs x t_max %d in ~15 s '
                         '(BASELINE.json configs[0]-sized batch), torch-CPU fp32 + NumPy preprocessing, %d threads; '
                         '%.0f ms per cycle' % (done, c_envs, T, cores, cms)}

    if rank == 0:
        line = {'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps,
                'warmup': max(args.warmup, 3), 'ms_per_step': ms_per_step, 'update_ms': ms_per_step,
                'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
                'dtype': {'fp32': 'f32', 'tf32x3': 'tf32x3', 'tf32': 'tf32', 'bf16x3': 'bf16x3'}[args.math], 'data': 'synthetic',
                'config': workload_config(args, world), 'clocks': clk, 'e2e': e2e, 'gpu_launches': int(launches),
                'roofline': roofline, 'cpu_baseline': cpu, 'variants': variants,
                'step_fraction_of_tensor_peak': step_frac, 'kernel_time_accounted': accounted / ms_total,
                'profiled_ms_per_step': ms_total / args.steps,
                'kernels': [{k: (round(v, 6) if isinstance(v, float) else v) for k, v in kk.items()} for kk in kernels],
                'loss': loss_val}
        if dumped:
            line['dumped_outputs'] = dumped
        print(json.dumps(line), flush=True)
    if world > 1:
        torch.distributed.destroy_process_group()


def main():
    args = parse()
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_b200(args)


if __name__ == '__main__':
    main()
