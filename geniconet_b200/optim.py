"""The optimizer step of the training loop as ONE kernel launch.

The reference trains with `torch.optim.Adam(model.parameters(), lr=...)` (run.py:446) and calls `optimizer.step()` once per batch
(run.py:250), optionally followed by a CyclicLR scheduler step (run.py:252-254).  `Adam` below is a `torch.optim.Optimizer`
with the same constructor arguments, the same per-parameter state (`step`, `exp_avg`, `exp_avg_sq` -- `step` an fp32 device
scalar as torch keeps it for capturable optimizers) and therefore an interchangeable `state_dict()`; its `step()` hands the
whole parameter list to `gin_adam_step` (geniconet_b200/csrc/gin_adam.cuh), which updates every tensor in one launch.

Safe under CUDA-graph capture: the tensor table lives in buffers allocated at construction, the step counters live on the
device, and a learning rate given as a device tensor (`lr=torch.tensor(1e-4, device=...)`, as torch requires for capturable
optimizers whose rate changes) is read at run time.  No CPU path: parameters must be CUDA fp32 tensors.
"""
import numpy as np
import torch

from . import _lib
from .ico_conv import _stream

_ROW = np.dtype([('p', '<u8'), ('g', '<u8'), ('m', '<u8'), ('v', '<u8'), ('step', '<u8'), ('n', '<i8')])      # GinAdamTensor


class Adam(torch.optim.Optimizer):
    """torch.optim.Adam (amsgrad=False, maximize=False) with a one-launch step; see the module docstring."""

    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0):
        if not isinstance(lr, torch.Tensor) and lr < 0.0:
            raise ValueError('Invalid learning rate: %r' % (lr,))
        if not 0.0 <= eps:
            raise ValueError('Invalid epsilon value: %r' % (eps,))
        if not 0.0 <= betas[0] < 1.0 or not 0.0 <= betas[1] < 1.0:
            raise ValueError('Invalid beta parameters: %r' % (betas,))
        if not 0.0 <= weight_decay:
            raise ValueError('Invalid weight_decay value: %r' % (weight_decay,))
        # the keys torch.optim.Adam keeps in a param group, so that state_dict()s are interchangeable
        defaults = dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay, amsgrad=False, maximize=False, foreach=None,
                        capturable=True, differentiable=False, fused=True, decoupled_weight_decay=False)
        super().__init__(params, defaults)
        self._chunk = None
        self._tables = {}

    _RING, _CAPTURE_SLOTS = 4, 2

    def _buffers(self, gi, group):
        """Per group, allocated once and never inside a capture: a ring of pinned host tables for eager steps (gradient tensors,
        hence the table, may change every step while earlier copies are still in flight), its device table, and a few
        (host, device) pairs reserved for CUDA-graph captures -- a captured copy node re-reads ITS pinned table on every replay,
        so that memory must never be rewritten."""
        if gi not in self._tables:
            n = len(group['params'])
            dev = group['params'][0].device
            nbytes = n * _ROW.itemsize + (n + 1) * 4
            new_host = lambda: torch.empty(nbytes, dtype=torch.uint8).pin_memory()
            new_dev = lambda: torch.zeros(nbytes, dtype=torch.uint8, device=dev)
            self._tables[gi] = {
                'rows_bytes': n * _ROW.itemsize, 'ticket': torch.zeros(1, dtype=torch.int32, device=dev),
                'ring': [{'host': new_host(), 'event': None} for _ in range(self._RING)], 'next': 0,
                'eager': {'dev': new_dev(), 'key': None, 'count': 0, 'chunks': 0},
                'captures': [{'host': new_host(), 'dev': new_dev(), 'key': None, 'count': 0, 'chunks': 0} for _ in range(self._CAPTURE_SLOTS)],
            }
        return self._tables[gi]

    def _fill(self, tb, host_t, rows):
        n = len(rows)
        host = host_t.numpy()
        host[:n * _ROW.itemsize].view(_ROW)[:] = np.array(rows, dtype=_ROW)
        chunks = np.array([(r[5] + self._chunk - 1) // self._chunk for r in rows], dtype=np.int64)
        first = np.zeros(n + 1, dtype=np.int32)
        first[1:] = np.cumsum(chunks)
        host[tb['rows_bytes']:tb['rows_bytes'] + (n + 1) * 4].view(np.int32)[:] = first
        return n, int(first[-1])

    def _table(self, tb, rows):
        """The device table holding `rows` (stream-ordered upload when it is not there yet)."""
        key = tuple(rows)
        if torch.cuda.is_current_stream_capturing():
            slot = next((c for c in tb['captures'] if c['key'] == key), None) or next((c for c in tb['captures'] if c['key'] is None), None)
            if slot is None:
                raise RuntimeError('geniconet_b200.optim.Adam: more than %d CUDA-graph captures with different parameter / gradient '
                                   'tensors; raise Adam._CAPTURE_SLOTS before the first step' % self._CAPTURE_SLOTS)
            if slot['key'] is None:
                slot['count'], slot['chunks'] = self._fill(tb, slot['host'], rows)
                slot['key'] = key
            slot['dev'].copy_(slot['host'], non_blocking=True)      # a copy node of THIS graph: nothing has executed yet
            return slot
        t = tb['eager']
        if key != t['key']:
            h = tb['ring'][tb['next']]
            tb['next'] = (tb['next'] + 1) % self._RING
            if h['event'] is not None:
                h['event'].synchronize()                           # the copy that last read this host table has run
            t['count'], t['chunks'] = self._fill(tb, h['host'], rows)
            t['dev'].copy_(h['host'], non_blocking=True)           # ordered after the previous step's kernel on this stream
            h['event'] = torch.cuda.Event()
            h['event'].record()
            t['key'] = key
        return t

    def _init_state(self, p):
        st = self.state[p]
        if len(st) == 0:
            if torch.cuda.is_current_stream_capturing():
                # tensors created inside a capture live in the graph's pool and would be re-zeroed by every replay
                raise RuntimeError('geniconet_b200.optim.Adam: optimizer state must exist before a CUDA-graph capture; '
                                   'call prepare() (or take one eager step) first')
            st['step'] = torch.zeros((), dtype=torch.float32, device=p.device)
            st['exp_avg'] = torch.zeros_like(p, memory_format=torch.preserve_format)
            st['exp_avg_sq'] = torch.zeros_like(p, memory_format=torch.preserve_format)
        elif not (isinstance(st['step'], torch.Tensor) and st['step'].is_cuda and st['step'].dtype == torch.float32):
            st['step'] = torch.as_tensor(float(st['step']), dtype=torch.float32, device=p.device)      # a state_dict written by a CPU-step Adam
        return st

    def prepare(self):
        """Allocate state and table buffers now (call before capturing a CUDA graph whose first step would otherwise do it)."""
        for gi, group in enumerate(self.param_groups):
            if group['params']:
                self._buffers(gi, group)
                for p in group['params']:
                    if p.requires_grad:
                        self._init_state(p)

    @torch.no_grad()
    def step(self, closure=None):
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        if self._chunk is None:
            self._chunk = int(_lib.lib.gin_adam_chunk())
        for gi, group in enumerate(self.param_groups):
            if group.get('amsgrad') or group.get('maximize') or group.get('decoupled_weight_decay'):
                raise NotImplementedError('geniconet_b200.optim.Adam: amsgrad / maximize / decoupled_weight_decay are not implemented')
            live = [p for p in group['params'] if p.grad is not None]
            if not live:
                continue
            rows = []
            for p in live:
                g = p.grad
                if not (p.is_cuda and p.dtype == torch.float32 and g.is_cuda and g.dtype == torch.float32):
                    raise RuntimeError('geniconet_b200.optim.Adam needs CUDA fp32 parameters and gradients (there is no CPU path)')
                if g.is_sparse:
                    raise RuntimeError('geniconet_b200.optim.Adam does not support sparse gradients')
                st = self._init_state(p)
                # one memory order for the four tensors: dense parameters only (contiguous in SOME format), gradient in the same one
                if not (p.is_contiguous() or p.is_contiguous(memory_format=torch.channels_last)):
                    raise RuntimeError('geniconet_b200.optim.Adam: parameter is not dense')
                if g.stride() != p.stride() and g.numel() > 1:
                    g = g.contiguous() if p.is_contiguous() else g.contiguous(memory_format=torch.channels_last)
                    p.grad = g
                if st['exp_avg'].stride() != p.stride() or st['exp_avg_sq'].stride() != p.stride():
                    raise RuntimeError('geniconet_b200.optim.Adam: optimizer state and parameter differ in memory layout')
                rows.append((p.data_ptr(), g.data_ptr(), st['exp_avg'].data_ptr(), st['exp_avg_sq'].data_ptr(), st['step'].data_ptr(), p.numel()))
            if gi not in self._tables and torch.cuda.is_current_stream_capturing():
                raise RuntimeError('geniconet_b200.optim.Adam: call prepare() (or take one eager step) before a CUDA-graph capture')
            tb = self._buffers(gi, group)
            t = self._table(tb, rows)
            lr = group['lr']
            lr_dev = 0
            if isinstance(lr, torch.Tensor):
                if lr.is_cuda:
                    if lr.dtype != torch.float32:
                        raise RuntimeError('geniconet_b200.optim.Adam: a tensor learning rate must be fp32')
                    lr_dev, lr = lr.data_ptr(), 0.0
                else:
                    lr = float(lr)
            b1, b2 = group['betas']
            _lib.check(_lib.lib.gin_adam_step(t['dev'].data_ptr(), t['dev'].data_ptr() + tb['rows_bytes'], t['count'], t['chunks'], float(lr), lr_dev,
                                              float(b1), float(b2), float(group['eps']), float(group['weight_decay']), tb['ticket'].data_ptr(), _stream()),
                       'gin_adam_step')
            # the kernel writes through raw pointers: bump the version counters as an in-place torch update would, so that caches
            # keyed on (data_ptr, _version) -- IcoConvS2S's packed weights -- see the new values
            for p in live:
                torch.autograd.graph.increment_version(p)
        return loss
