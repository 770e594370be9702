"""RolloutEngine: the device-resident half of PAACLearner.train() (paac.py:99-168).

It owns every device buffer one learner needs for N environments and t_max steps and issues the C-ABI
calls in the order the reference's loop implies:

    for t in range(T):   act(t)      -> paacb_policy_forward_sample (forward + in-kernel Philox sampling)   paac.py:105-112
                         observe(t)  -> paacb_observe_u8 (K1 + reward / episode-over bookkeeping)          emulator_runner.py:24-31,
                                                                                                           paac.py:119-123
    update(lr)           -> bootstrap forward (paac.py:140-142), training forward, paacb_returns_loss_grad
                            (paac.py:144-149 + the loss graph), paacb_backward, [NCCL allreduce],
                            paacb_clip_rmsprop (actor_learner.py:54-70)

All launches go to the current torch stream without host synchronisation.  PyTorch is used for memory, streams,
CUDA-graph capture and torch.distributed only: no torch kernel runs inside a rollout-and-update cycle.

Rollout states.  The reference keeps states[T, N, 84, 84, 4] and re-reads the shared buffer for the next rollout
(paac.py:92,112).  Here two rollouts' worth of states ping-pong: rollout c lives in half c & 1 (slots 0..T-1 contiguous:
the training batch is one [T*N, 84, 84, 4] tensor, paac.py:151) and its LAST state s_T is written straight into slot 0
of the other half, where it is both the bootstrap state (paac.py:140) and the first state of rollout c + 1.  Nothing is
copied between rollouts (the first version copied 116 MB per update at 4096 envs).  ``state(t)`` is the view of s_t.

Scheduling of the training forward (``train_forward=``).  PAAC's training batch is the concatenation of the t_max
acting batches under unchanged parameters (paac.py:92,112,151), so its forward can be scheduled three ways with
bit-identical results (tests/test_gpu_learner.py):
    'batched'   the reference's schedule: one forward over T*N samples inside update()               (default)
    'stepwise'  the SAME work issued per step with ``train_forward_step(t)`` (paacb_policy_forward_at), e.g. while the
                emulators run and the frames cross PCIe; update() issues whatever steps are still missing
    'reuse'     act(t) writes its activations straight into the training workspace and update() runs no training
                forward at all (the acting forward already IS that computation); values[t] aliases v

CUDA graphs (``enable_graphs()``; the reference's default is 32 environments, train.py:95, where a cycle is ~60 small
launches and launch latency is the whole cost).  act(t), train_forward_step(t) and update() are then captured once per
ping-pong half and replayed: one graph launch each.  What changes between replays lives in device memory, not in
kernel arguments: the learning rate (paacb_clip_rmsprop_dlr), the Philox draw base (paacb_rng_advance) and the
optimizer's self-resetting grid barrier.  Results are bit-identical to the eager calls (tests/test_gpu_graphs.py).
"""
import ctypes as C

import numpy as np
import torch

from . import _lib, parallel

STATE_SHAPE = (84, 84, 4)
FRAME_SLOT_SHAPE = (4, 2, 210, 160)
MAX_T = 64            # kLossMaxT in csrc/loss.cu: the returns + loss kernel keeps 5 * 32 floats per time step in shared memory


class RolloutEngine(object):

    def __init__(self, network, n_envs, t_max, gamma=0.99, rho=0.99, eps=0.1, momentum=0.0,
                 clip_norm=3.0, clip_norm_type='global', seed=3, process_group=None, world_size=1,
                 train_forward='batched', overlap_allreduce=True, sampling='philox', first_env=0):
        self.net = network
        self.lib = network._lib
        self.ctx = network.ctx
        self.dev = network.torch_device
        self.N, self.T, self.A = int(n_envs), int(t_max), int(network.num_actions)
        if self.T > MAX_T:
            # refused here rather than by paacb_returns_loss_grad at the end of the first rollout
            raise ValueError('t_max %d exceeds %d, the longest rollout the returns + loss kernel supports' % (self.T, MAX_T))
        self.B = self.N * self.T
        self.gamma, self.rho, self.eps, self.momentum = float(gamma), float(rho), float(eps), float(momentum)
        self.clip_norm = float(clip_norm)
        if clip_norm_type == 'global':
            self.clip_type = _lib.CLIP_GLOBAL
        elif clip_norm_type == 'ignore':
            self.clip_type = _lib.CLIP_IGNORE
        elif clip_norm_type == 'local':
            raise Exception("clip_norm_type 'local' is broken in the reference (actor_learner.py:62-63 iterates "
                            "(grad, var) tuples); use 'global' or 'ignore'")
        else:
            raise Exception('Norm type not recognized')          # actor_learner.py:67
        if sampling not in ('philox', 'injected'):
            raise ValueError("sampling must be 'philox' (uniforms drawn inside the heads kernel) or 'injected' "
                             "(the caller fills engine.uniforms)")
        self.sampling = sampling
        self.first_env = int(first_env)       # global index of this learner's first environment (multi-GPU: rank * N)
        self.beta = float(network.entropy_regularisation_strength)
        self.group, self.world = process_group, int(world_size)
        self.overlap_allreduce = bool(overlap_allreduce)
        self.tail_off = int(self.lib.paacb_grad_tail_offset(self.ctx))
        self._pending = []
        self.tail_group = self.group
        if self.world > 1 and self.overlap_allreduce and hasattr(self.lib, 'paacb_set_sm_reserve'):
            # The tail's all-reduce runs under the conv weight-gradient kernels, which are persistent CTAs with the maximum
            # shared-memory carve-out: they leave PAACB_SM_RESERVE SMs free, and the collective must FIT there.  NCCL's default on
            # NVSwitch is up to 24 NVLS channels = 24 CTAs that all have to be resident before any of them makes progress: with 8 SMs
            # free, 8 of them spin until the first weight-gradient kernel retires, the other 16 then take SMs from the NEXT kernel,
            # whose last 16 CTAs wait for the collective and run alone afterwards (measured at 8 GPUs: conv2's weight gradient
            # 0.31 -> 0.47 ms, the whole cost of the N = 8 step over the N = 1 step).  So the tail goes through its own
            # communicator limited to as many CTAs as SMs are reserved (ProcessGroupNCCL max_ctas; 6.4 MB on 8 CTAs: 94 us
            # against 71 us on 24, tools/experiments/allreduce_probe.py); the small conv-head reduction after the backward
            # keeps the default communicator.
            import os
            reserve = int(os.environ.get('PAACB_SM_RESERVE', '8'))
            _lib.check(self.lib.paacb_set_sm_reserve(self.ctx, reserve), 'paacb_set_sm_reserve')
            max_ctas = int(os.environ.get('PAACB_TAIL_MAX_CTAS', str(reserve)))
            if max_ctas > 0 and torch.distributed.get_backend(self.group) == 'nccl':
                opts = torch.distributed.ProcessGroupNCCL.Options()
                opts.config.max_ctas = max_ctas
                opts.config.min_ctas = 1
                ranks = torch.distributed.get_process_group_ranks(self.group) if self.group is not None else list(range(self.world))
                self.tail_group = torch.distributed.new_group(ranks=ranks, pg_options=opts)

        d, N, T, A, B = self.dev, self.N, self.T, self.A, self.B
        f32 = dict(dtype=torch.float32, device=d)
        self._sbuf = torch.zeros((2, T, N) + STATE_SHAPE, dtype=torch.uint8, device=d)      # ping-pong rollout states
        self._cur = 0
        self.actions = torch.zeros((T, N), dtype=torch.int32, device=d)
        self.onehot = torch.zeros((N, A), **f32)
        self.values = torch.zeros((T, N), **f32)
        self.rewards = torch.zeros((T, N), **f32)
        self.over = torch.zeros((T, N), **f32)
        self.uniforms = torch.zeros((T, N), **f32)       # sampling='injected' only
        self.pi_act = torch.zeros((N, A), **f32)
        self.boot_v = torch.zeros((N,), **f32)
        self.boot_pi = torch.zeros((N, A), **f32)
        self.pi = torch.zeros((B, A), **f32)
        self.v = torch.zeros((B,), **f32)
        self.y = torch.zeros((B,), **f32)
        self.adv = torch.zeros((B,), **f32)
        self.dlogits = torch.zeros((B, A), **f32)
        self.dv = torch.zeros((B,), **f32)
        self.loss = torch.zeros((1,), **f32)
        self.norm = torch.zeros((1,), **f32)
        P = network.param_count
        self.grads = torch.zeros((P,), **f32)
        self.ms = torch.ones((P,), **f32)            # rms slot <- ones, momentum slot <- zeros (SURVEY App. B)
        self.mom = torch.zeros((P,), **f32)
        self.act_ws = torch.empty((network.workspace_floats(N),), **f32)
        self.fwd_ws = torch.empty((network.workspace_floats(B),), **f32)
        self.bwd_ws = torch.empty((int(self.lib.paacb_backward_workspace_floats(self.ctx, B)),), **f32)
        self.opt_ws = torch.empty((int(self.lib.paacb_optimizer_workspace_floats(self.ctx)),), **f32)
        # Philox state in device memory: {seed, draw base}; one draw index per env step (paacb_policy_forward_sample)
        self.rng = torch.tensor([int(seed), 0], dtype=torch.int64, device=d)
        self.lr_dev = torch.zeros((1,), **f32)       # the learning rate a replayed update graph reads
        self._lr_host = torch.zeros((1,), dtype=torch.float32)
        if d.type == 'cuda':
            self._lr_host = self._lr_host.pin_memory()
        self.gen = torch.Generator(device=d)         # sampling='injected': draw_uniforms()
        self.gen.manual_seed(int(seed))
        self._slice_ws = {}        # forward workspaces of environment slices (act(t, lo, hi))
        self._stepped = set()      # (t, lo, hi) slices of the training forward already issued ('stepwise')
        self._booted = []          # [lo, hi) slices whose bootstrap value V(s_T) was already issued (bootstrap())
        self._values_own = self.values
        self._graphs = None        # enable_graphs(): {key: torch.cuda.CUDAGraph}
        self.set_train_forward(train_forward)

    # ---- rollout states ---------------------------------------------------------------------------
    def state(self, t):
        """View of s_t, t in [0, T]: uint8 [N, 84, 84, 4].  s_T lives in slot 0 of the other half (it is s_0 of the next rollout)."""
        return self._sbuf[self._cur, t] if t < self.T else self._sbuf[1 - self._cur, 0]

    @property
    def flat_states(self):
        """The training batch [T*N, 84, 84, 4] (paac.py:151)."""
        return self._sbuf[self._cur].view((self.B,) + STATE_SHAPE)

    def set_states(self, states):
        """states: [T+1, N, 84, 84, 4] (or [1, ...] for s_0 alone), tensor or array."""
        states = torch.as_tensor(states)
        for t in range(states.shape[0]):
            self.state(t).copy_(states[t])

    def get_states(self):
        """Copy of s_0 .. s_T as one [T+1, N, 84, 84, 4] tensor."""
        return torch.stack([self.state(t) for t in range(self.T + 1)])

    # ---- helpers ----------------------------------------------------------------------------------
    def set_train_forward(self, mode):
        """Choose the schedule of the training forward (see the module docstring); call between updates only."""
        if mode not in ('batched', 'stepwise', 'reuse'):
            raise ValueError("train_forward must be 'batched', 'stepwise' or 'reuse'")
        if getattr(self, '_graphs', None):
            self._graphs.clear()                # captured graphs embed the schedule
        self.train_forward = mode
        self._stepped.clear()
        # 'reuse': the acting value IS the training value
        self.values = self.v.view(self.T, self.N) if mode == 'reuse' else self._values_own

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.dev).cuda_stream)

    def draw_uniforms(self):
        """sampling='injected': one torch draw per update for all T*N sampling decisions into ``uniforms``.
        sampling='philox' (default): nothing to do, the heads kernel draws its own uniforms (kept so that callers written for
        the injected mode run unchanged)."""
        if self.sampling != 'injected':
            return
        self.uniforms.uniform_(0.0, 1.0, generator=self.gen)
        # uniform_ on fp32 can return exactly 1.0 only by rounding; keep u in [0, 1)
        self.uniforms.clamp_(max=float(np.nextafter(np.float32(1.0), np.float32(0.0))))

    def _sample_args(self, t, lo, hi):
        if self.sampling == 'injected':
            return dict(uniforms=self.uniforms[t, lo:hi])
        return dict(rng=self.rng, draw=t, first_sample=self.first_env + lo)

    # ---- CUDA graphs ------------------------------------------------------------------------------
    def enable_graphs(self):
        """Capture act / train_forward_step / update as CUDA graphs on first use and replay them afterwards.
        Runs one eager warm-up cycle first (kernel attributes and lazily allocated workspaces must exist before a capture)
        and restores parameters, optimizer slots and the Philox state afterwards, so the call has no numerical effect."""
        if self.world > 1 and self.overlap_allreduce:
            self.overlap_allreduce = False          # graphed update: [graph: ... backward] -> all-reduce -> [graph: optimizer]
        keep = [t.clone() for t in (self.net.params, self.ms, self.mom, self.rng, self.rewards, self.over, self._values_own)]
        for t in range(self.T):
            self.act(t)
            if self.train_forward == 'stepwise':
                self.train_forward_step(t)
        self.update(0.0, roll=False)
        for dst, src in zip((self.net.params, self.ms, self.mom, self.rng, self.rewards, self.over, self._values_own), keep):
            dst.copy_(src)
        self.net.params_changed()
        self.net.forward(self.state(0), self.pi_act, self.boot_v, self.act_ws)      # rebuild the cached weight images now
        torch.cuda.synchronize(self.dev)
        self._graphs = {}

    def _run(self, key, fn):
        """fn() eagerly, or -- with graphs enabled -- the captured graph of fn() for this (call, ping-pong half)."""
        if self._graphs is None:
            return fn()
        key = key + (self._cur,)
        g = self._graphs.get(key)
        if g is None:
            g = torch.cuda.CUDAGraph()
            side = torch.cuda.Stream(self.dev)
            side.wait_stream(torch.cuda.current_stream(self.dev))
            with torch.cuda.graph(g, stream=side):
                fn()
            self._graphs[key] = g
        g.replay()

    # ---- rollout ----------------------------------------------------------------------------------
    def act(self, t, lo=0, hi=None, onehot_out=None):
        """Forward on s_t + categorical sampling; fills actions[t], values[t], onehot, pi_act.
        [lo, hi) restricts the call to a contiguous slice of the environments (the runner protocol hands every worker
        a contiguous slice, runners.py:17-18): slices can be issued on different streams so that the next slice's
        forward overlaps this slice's frame ingestion.
        onehot_out: (tensor-like with data_ptr) destination of the one-hot actions instead of ``onehot`` -- e.g. the
        runners' shared action array in pinned, mapped host memory (paac.py:107-108 without a copy)."""
        if hi is None:
            hi = self.N
        self._run(('act', t, lo, hi, 0 if onehot_out is None else int(onehot_out.data_ptr())),
                  lambda: self._act(t, lo, hi, onehot_out))

    def _act(self, t, lo, hi, onehot_out):
        oh = self.onehot[lo:hi] if onehot_out is None else onehot_out
        if self.train_forward == 'reuse':
            first = t * self.N + lo
            self.net.forward(self.state(t)[lo:hi], self.pi[first:first + hi - lo], self.v[first:first + hi - lo], self.fwd_ws,
                             actions=self.actions[t, lo:hi], onehot=oh, ws_capacity=self.B, ws_first=first,
                             **self._sample_args(t, lo, hi))
            return
        self.net.forward(self.state(t)[lo:hi], self.pi_act[lo:hi], self.values[t, lo:hi], self._ws_for(lo, hi),
                         actions=self.actions[t, lo:hi], onehot=oh, **self._sample_args(t, lo, hi))

    def observe_frames(self, t, frames_ptr, pairs_per_env, reset_u8, rewards, over, lo=0, hi=None, over_is_reset=False):
        """Raw-frame protocol: s_{t+1} <- preprocess(frames | s_t), rewards[t] / over[t] <- the step's reward and episode-over
        flag, ONE launch (paacb_observe_u8).  rewards / over: float32 [N] device tensors, or tensors over pinned, mapped host
        memory (anything with .data_ptr() the GPU can read).  frames_ptr addresses the slot of environment `lo`; it may point
        into pinned, mapped HOST memory (the kernel then reads the rows it needs zero-copy over PCIe).
        over_is_reset: over[n] != 0 also resets environment n's stack (emulator_runner.py:26-27; needs 4 pairs per env)."""
        if hi is None:
            hi = self.N
        p = _lib.ptr
        f4 = 4
        rin = rewards.data_ptr() + (lo * f4 if rewards.shape[0] == self.N else 0)
        oin = over.data_ptr() + (lo * f4 if over.shape[0] == self.N else 0)
        _lib.check(self.lib.paacb_observe_u8(self.ctx, C.c_void_p(frames_ptr), int(pairs_per_env),
                                             p(reset_u8[lo:hi]) if reset_u8 is not None else None,
                                             p(self.state(t)[lo:hi]), p(self.state(t + 1)[lo:hi]), hi - lo,
                                             C.c_void_p(rin), C.c_void_p(oin), p(self.rewards[t, lo:hi]), p(self.over[t, lo:hi]),
                                             1 if over_is_reset else 0, self._stream()), 'paacb_observe_u8')

    def observe_states(self, t, states, rewards, over):
        """Classic protocol: the environments produced stacked 84x84x4 observations themselves."""
        self.state(t + 1).copy_(states, non_blocking=True)
        self.rewards[t].copy_(rewards, non_blocking=True)
        self.over[t].copy_(over, non_blocking=True)

    def _ws_for(self, lo, hi):
        if lo == 0 and hi == self.N:
            return self.act_ws
        ws = self._slice_ws.get((lo, hi))
        if ws is None:
            ws = self._slice_ws[(lo, hi)] = torch.empty((self.net.workspace_floats(hi - lo),), dtype=torch.float32,
                                                        device=self.dev)
        return ws

    def bootstrap(self, lo=0, hi=None):
        """V(s_T) of a slice of the environments (paac.py:140-142), as soon as ITS last frames are in: the end-to-end loop
        issues it per slice so that it overlaps the frame ingestion of the other slices.  update() computes the bootstrap
        of whatever slices were not issued."""
        if hi is None:
            hi = self.N
        self.net.forward(self.state(self.T)[lo:hi], self.boot_pi[lo:hi], self.boot_v[lo:hi], self._ws_for(lo, hi))
        self._booted.append((lo, hi))

    def train_forward_step(self, t, lo=0, hi=None):
        """'stepwise': the training forward of the samples (t, lo..hi), written into their place in the batch workspace."""
        if self.train_forward != 'stepwise':
            raise RuntimeError("train_forward_step() needs RolloutEngine(train_forward='stepwise')")
        if hi is None:
            hi = self.N
        self._run(('tfs', t, lo, hi), lambda: self._train_forward_step(t, lo, hi))
        self._stepped.add((t, lo, hi))

    def _train_forward_step(self, t, lo, hi):
        first = t * self.N + lo
        self.net.forward(self.state(t)[lo:hi], self.pi[first:first + hi - lo], self.v[first:first + hi - lo], self.fwd_ws,
                         ws_capacity=self.B, ws_first=first)

    def _missing_steps(self):
        """The (t, lo, hi) pieces of the training forward the caller has not issued itself (whole steps or the gaps)."""
        out = []
        for t in range(self.T):
            covered = sorted((lo, hi) for (tt, lo, hi) in self._stepped if tt == t)
            pos = 0
            for lo, hi in covered:
                if lo > pos:
                    out.append((t, pos, lo))
                pos = max(pos, hi)
            if pos < self.N:
                out.append((t, pos, self.N))
        return out

    def _finish_stepwise(self):
        for t, lo, hi in self._missing_steps():
            self.train_forward_step(t, lo, hi)
        self._stepped.clear()

    # ---- update -----------------------------------------------------------------------------------
    def _missing_bootstraps(self):
        out, pos = [], 0
        for lo, hi in sorted(self._booted):
            if lo > pos:
                out.append((pos, lo))
            pos = max(pos, hi)
        if pos < self.N:
            out.append((pos, self.N))
        return out

    def forward_backward(self):
        """Bootstrap forward, training forward, returns + loss gradient, backward.  Leaves dL/dparams in grads."""
        boots = tuple(self._missing_bootstraps())                                                 # paac.py:140-142
        steps = tuple(self._missing_steps()) if self.train_forward == 'stepwise' else ()
        self._booted = []
        self._stepped.clear()
        overlap = self.world > 1 and self.overlap_allreduce
        if overlap:
            self._forward_backward(boots, steps, True)
        else:
            self._run(('fb', boots, steps), lambda: self._forward_backward(boots, steps, False))

    def _forward_backward(self, boots, steps, overlap):
        T, N, B = self.T, self.N, self.B
        p = _lib.ptr
        st = self._stream()
        for lo, hi in boots:
            self.net.forward(self.state(T)[lo:hi], self.boot_pi[lo:hi], self.boot_v[lo:hi], self._ws_for(lo, hi))
        flat_states = self.flat_states                                                            # paac.py:151
        if self.train_forward == 'batched':
            self.net.forward(flat_states, self.pi, self.v, self.fwd_ws)
        for t, lo, hi in steps:
            self._train_forward_step(t, lo, hi)
        _lib.check(self.lib.paacb_returns_loss_grad(
            self.ctx, p(self.rewards), p(self.over), p(self.values), p(self.boot_v), p(self.actions), p(self.pi),
            p(self.v), T, N, C.c_double(self.gamma), C.c_float(self.beta), p(self.y), p(self.adv), p(self.dlogits),
            p(self.dv), p(self.loss), st), 'paacb_returns_loss_grad')
        if overlap:
            # multi-GPU: the tail of the flat gradient (hidden fc layer + heads, 95 % of the parameters) is final after the
            # first part of the backward; its all-reduce runs on NCCL's stream under the conv layers' weight gradients
            for part in (_lib.BWD_TAIL, _lib.BWD_HEAD):
                _lib.check(self.lib.paacb_backward_part(self.ctx, p(self.net.params), p(flat_states), B, p(self.fwd_ws),
                                                        p(self.dlogits), p(self.dv), p(self.bwd_ws), p(self.grads), part, st),
                           'paacb_backward_part')
                if part == _lib.BWD_TAIL:
                    self._pending = [torch.distributed.all_reduce(self.grads[self.tail_off:], op=torch.distributed.ReduceOp.SUM,
                                                                  group=self.tail_group, async_op=True)]
            return
        _lib.check(self.lib.paacb_backward(self.ctx, p(self.net.params), p(flat_states), B, p(self.fwd_ws),
                                           p(self.dlogits), p(self.dv), p(self.bwd_ws), p(self.grads), st),
                   'paacb_backward')

    def allreduce(self):
        if self.world > 1:
            if self._pending:
                self._pending.append(torch.distributed.all_reduce(self.grads[:self.tail_off], op=torch.distributed.ReduceOp.SUM,
                                                                  group=self.group, async_op=True))
                for w in self._pending:
                    w.wait()             # stream-level wait: the optimizer kernel is ordered after both reductions
                self._pending = []
            else:
                parallel.allreduce_mean_grads(self.grads, self.world, self.group)

    def apply(self, lr):
        """Global-norm clip + RMSProp (+ refresh of the cached weight images) and the Philox draw base += T."""
        if self._graphs is not None:
            self._lr_host[0] = float(lr)
            self.lr_dev.copy_(self._lr_host, non_blocking=True)      # an H2D memcpy, not a kernel
        self._run(('apply',), lambda: self._apply(lr))

    def _apply(self, lr):
        p = _lib.ptr
        common = (C.c_float(self.rho), C.c_float(self.eps), C.c_float(self.momentum), C.c_float(self.clip_norm),
                  self.clip_type, p(self.norm), p(self.opt_ws), self._stream())
        if self._graphs is not None:
            _lib.check(self.lib.paacb_clip_rmsprop_dlr(self.ctx, p(self.net.params), p(self.ms), p(self.mom), p(self.grads),
                                                       C.c_float(1.0 / self.world), p(self.lr_dev), *common),
                       'paacb_clip_rmsprop_dlr')
        else:
            _lib.check(self.lib.paacb_clip_rmsprop(self.ctx, p(self.net.params), p(self.ms), p(self.mom), p(self.grads),
                                                   C.c_float(1.0 / self.world), C.c_float(lr), *common), 'paacb_clip_rmsprop')
        if self.sampling == 'philox':
            _lib.check(self.lib.paacb_rng_advance(self.ctx, p(self.rng), self.T, self._stream()), 'paacb_rng_advance')

    def roll(self):
        """The last state of this rollout is the first state of the next (paac.py:99-112 reuse shared_states): it already
        lies in slot 0 of the other half -- flip halves, copy nothing."""
        self._cur ^= 1

    def update(self, lr, roll=True):
        self.forward_backward()
        self.allreduce()
        self.apply(lr)
        if roll:
            self.roll()
