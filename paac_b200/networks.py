"""Network / NIPSNetwork / NatureNetwork: host-side mirror of the reference's networks.py:100-169.

Same class names, same ``conf`` dict keys, same attribute names (``input_ph``, ``selected_action_ph``,
``loss_scaling``, ``output``, ...), same composition by multiple inheritance.  Where the reference builds a
TF1 graph, these classes create a ``paacb`` context (the C-ABI extension, include/paacb.h) and own the flat
fp32 parameter buffer on the GPU.  The "placeholders" are small handle objects that the ``Session`` shim
(paac_b200/session.py) understands, so reference-style ``session.run([...], feed_dict={...})`` code works.

There is no CPU path: ``conf['device']`` must name a GPU ('/gpu:K', as train.py:80 defaults).
"""
import ctypes as C
import logging
import os
import re

import numpy as np
import torch

from . import _lib


class Placeholder(object):
    """Stand-in for a tf.placeholder (networks.py:113-114): a hashable feed_dict key."""

    def __init__(self, name, dtype, shape):
        self.name, self.dtype, self.shape = name, dtype, shape

    def __repr__(self):
        return 'Placeholder(%s, %s, %s)' % (self.name, self.dtype, self.shape)


class Fetch(object):
    """Stand-in for a fetchable tf.Tensor / tf.Operation of the reference graph."""

    def __init__(self, owner, kind):
        self.owner, self.kind = owner, kind

    def __repr__(self):
        return 'Fetch(%s)' % self.kind


def parse_device(device):
    """'/gpu:1' -> torch.device('cuda', 1).  '/cpu:0' is refused: the product has no CPU path."""
    m = re.match(r'^/?(gpu|cuda):(\d+)$', str(device).lower())
    if not m:
        raise _lib.PaacbError("device %r: this implementation runs on B200 GPUs only ('/gpu:K'); "
                              "the CPU restatement lives in oracle/ for tests" % (device,))
    return torch.device('cuda', int(m.group(2)))


class Network(object):

    ARCH = None      # set by NIPSNetwork / NatureNetwork

    def __init__(self, conf):
        self.name = conf['name']
        self.num_actions = conf['num_actions']
        self.clip_norm = conf['clip_norm']
        self.clip_norm_type = conf['clip_norm_type']
        self.device = conf['device']
        self.math = conf.get('math', 'fp32')
        self.seed = conf.get('seed', None)

        self.loss_scaling = 5.0
        self.input_ph = Placeholder('input', np.uint8, [None, 84, 84, 4])
        self.selected_action_ph = Placeholder('selected_action', np.float32, [None, self.num_actions])
        # networks.py:115 -- the 1/255 scaling is fused into the first conv's operand load (gemm_simt.cu)
        self.input = Fetch(self, 'input')

        # This class should never be used, must be subclassed
        self.output = None

    # ---- B200 side: context + parameters ----------------------------------------------------------
    def _create_context(self):
        lib = _lib.load()
        self.torch_device = parse_device(self.device)
        if not torch.cuda.is_available():
            raise _lib.PaacbError('no CUDA device visible: the PAAC B200 path has no CPU fallback')
        torch.cuda.set_device(self.torch_device)
        torch.cuda.init()
        handle = C.c_void_p()
        arch = _lib.ARCH_NIPS if self.ARCH == 'NIPS' else _lib.ARCH_NATURE
        _lib.check(lib.paacb_create(C.byref(handle), arch, int(self.num_actions), self.torch_device.index),
                   'paacb_create')
        self._lib, self.ctx = lib, handle
        self.set_math(self.math)
        self.param_count = int(lib.paacb_param_count(self.ctx))
        self.tensors = []        # (name, offset, shape, fan_in) in TF variable-creation order
        for i in range(lib.paacb_num_tensors(self.ctx)):
            name = C.create_string_buffer(64)
            off, nd, fan = C.c_int64(), C.c_int(), C.c_int64()
            shp = (C.c_int64 * 4)()
            _lib.check(lib.paacb_tensor_info(self.ctx, i, name, 64, C.byref(off), C.byref(nd), C.byref(shp),
                                             C.byref(fan)), 'paacb_tensor_info')
            self.tensors.append((name.value.decode(), off.value, tuple(shp[k] for k in range(nd.value)), fan.value))
        self.params = torch.empty(self.param_count, dtype=torch.float32, device=self.torch_device)
        self.initialize(self.seed)

    def set_math(self, math):
        """'fp32' (SIMT FFMA, the parity anchor: what the reference's fp32 graph computes, <= 2e-6 of it) | 'bf16x3' (tensor cores
        on bf16-split operands, hi*hi + hi*lo + lo*hi with fp32 accumulation: <= 2.5e-5 of the fp64 oracle through the whole
        network, inside the 1e-4 parity bar, both architectures) | 'tf32x3' (tensor cores on tf32-split operands, the first
        tensor-core generation: parity grade, 3x slower) | 'tf32' (plain tf32, 2e-4 .. 8e-4: a speed mode, NOT parity grade) |
        'auto' = 'bf16x3'."""
        if str(math).lower() == 'auto':
            math = 'bf16x3'
        mode = {'fp32': _lib.MATH_FP32, 'tf32x3': _lib.MATH_TF32X3, 'tf32': _lib.MATH_TF32,
                'bf16x3': _lib.MATH_BF16X3}[str(math).lower()]
        _lib.check(self._lib.paacb_set_math(self.ctx, mode), 'paacb_set_math')
        self.math = str(math).lower()

    def initialize(self, seed=None):
        """'torch' init of networks.py:24-46,63-81: U(-d, d), d = 1/sqrt(fan_in), weights AND biases."""
        rng = np.random.RandomState(seed)
        flat = np.empty(self.param_count, np.float32)
        for name, off, shape, fan in self.tensors:
            d = 1.0 / np.sqrt(fan)
            n = int(np.prod(shape))
            flat[off:off + n] = rng.uniform(-d, d, size=n).astype(np.float32)
        self.params.copy_(torch.from_numpy(flat))
        self.params_changed()

    def params_changed(self):
        """Tell the library that the parameter buffer was written from outside (it caches operand images of the weights
        between forwards; paacb_clip_rmsprop refreshes them itself).  Call after ANY direct write to ``params`` /
        ``variable(name)``."""
        _lib.check(self._lib.paacb_params_changed(self.ctx), 'paacb_params_changed')

    def variable(self, name):
        """View of one variable inside the flat buffer (reference layout: HWIO / [in, out]).
        After WRITING through such a view call ``params_changed()``: the library caches operand images of the weights."""
        for n, off, shape, _ in self.tensors:
            if n == name:
                return self.params[off:off + int(np.prod(shape))].view(*shape)
        raise KeyError(name)

    def variables(self):
        return {n: self.variable(n) for n, _, _, _ in self.tensors}

    def set_params(self, flat):
        self.params.copy_(torch.as_tensor(np.asarray(flat, np.float32)).reshape(-1))
        self.params_changed()

    def get_params(self):
        return self.params.detach().cpu().numpy().copy()

    LAYER_SHAPES = None      # per-sample shapes of the workspace activations, set by the subclasses

    def layer_tensors(self, ws, batch):
        """Per-layer fp32 views/copies [batch, ...] of a forward (activations) or backward (dZ) workspace.
        fp32 / tf32 modes store floats; 'bf16x3' stores each tensor as two bf16 planes, value = hi + lo."""
        out, off = [], 0
        raw = ws.view(torch.uint8)
        for shp in self.LAYER_SHAPES:
            e = int(np.prod(shp)) * batch
            if self.math == 'bf16x3':
                hi = raw[off * 4: off * 4 + e * 2].view(torch.bfloat16).float()
                lo = raw[off * 4 + e * 2: off * 4 + e * 4].view(torch.bfloat16).float()
                out.append((hi + lo).view((batch,) + tuple(shp)))
            else:
                out.append(ws[off:off + e].view((batch,) + tuple(shp)))
            off += e
        return out

    def workspace_floats(self, batch):
        return int(self._lib.paacb_forward_workspace_floats(self.ctx, int(batch)))

    def forward(self, states, pi, v, ws, uniforms=None, actions=None, onehot=None, ws_capacity=None, ws_first=0,
                rng=None, draw=0, first_sample=0):
        """Asynchronous forward on the current torch stream; all arguments are CUDA tensors.
        ws_capacity / ws_first: write samples [ws_first, ws_first + b) of a workspace laid out for ws_capacity samples.
        Sampling: ``uniforms`` (float32 [b], injected) or ``rng`` (int64 [2] device tensor {seed, draw base}: the heads kernel
        draws Philox uniforms itself for draw index ``draw`` and global sample indices first_sample .. first_sample + b)."""
        b = states.shape[0]
        st = C.c_void_p(torch.cuda.current_stream(self.torch_device).cuda_stream)
        p = _lib.ptr
        cap = b if ws_capacity is None else int(ws_capacity)
        if rng is not None:
            _lib.check(self._lib.paacb_policy_forward_sample(self.ctx, p(self.params), p(states), b, p(ws), cap, int(ws_first),
                                                             p(pi), p(v), p(rng), int(draw), int(first_sample), p(actions),
                                                             p(onehot), st), 'paacb_policy_forward_sample')
            return
        _lib.check(self._lib.paacb_policy_forward_at(self.ctx, p(self.params), p(states), b, p(ws), cap, int(ws_first),
                                                     p(pi), p(v), p(uniforms), p(actions), p(onehot), st),
                   'paacb_policy_forward_at')

    def launch_count(self):
        return int(self._lib.paacb_launch_count(self.ctx))

    def __del__(self):
        try:
            if getattr(self, 'ctx', None):
                self._lib.paacb_destroy(self.ctx)
                self.ctx = None
        except Exception:
            pass

    # ---- reference API: networks.py:122-135 -------------------------------------------------------
    def init(self, checkpoint_folder, saver, session):
        last_saving_step = 0
        path = saver.latest_checkpoint(checkpoint_folder) if saver is not None else None
        if path is None:
            logging.info('Initializing all variables')
        else:
            logging.info('Restoring network variables from previous run')
            saver.restore(session, path)
            last_saving_step = int(path[path.rindex('-') + 1:].split('.')[0])
        return last_saving_step


class NIPSNetwork(Network):
    """networks.py:138-151: 84x84x4 -conv8/4-> 20x20x16 -conv4/2-> 9x9x32 -> fc 256."""
    ARCH = 'NIPS'
    LAYER_SHAPES = [(20, 20, 16), (9, 9, 32), (256,)]

    def __init__(self, conf):
        super(NIPSNetwork, self).__init__(conf)
        self.output = Fetch(self, 'fc3')


class NatureNetwork(Network):
    """networks.py:154-169: -conv8/4-> 20x20x32 -conv4/2-> 9x9x64 -conv3/1-> 7x7x64 -> fc 512."""
    ARCH = 'NATURE'
    LAYER_SHAPES = [(20, 20, 32), (9, 9, 64), (7, 7, 64), (512,)]

    def __init__(self, conf):
        super(NatureNetwork, self).__init__(conf)
        self.output = Fetch(self, 'fc4')
