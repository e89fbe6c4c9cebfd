"""``Adam`` with torch.optim.Adam's constructor, semantics and state_dict layout, stepping through
``cpc_adam_step``: one kernel updates every parameter tensor (SURVEY.md 8(f) row 4, "fused Adam").

The trainer receives the optimizer *class* (contrastive_estimation_training.py:41, ``optimizer=torch.optim.Adam``)
and instantiates it as ``optimizer(model.parameters(), lr=lr)`` (:84); ``ContrastiveEstimationTrainer`` swaps in
this class when it is handed ``torch.optim.Adam`` and the model lives on a GPU.  The step count is a device
scalar, so the optimizer can be captured into a CUDA graph as is.
"""
import ctypes

import torch

from . import _lib, ops


class Adam(torch.optim.Optimizer):
    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0., amsgrad=False, maximize=False,
                 **unused):
        if amsgrad:
            raise _lib.CpcError("cpc_b200.optim.Adam: amsgrad is not implemented (the reference never sets it)")
        if lr < 0 or eps < 0 or not 0 <= betas[0] < 1 or not 0 <= betas[1] < 1 or weight_decay < 0:
            raise ValueError("invalid Adam hyper-parameters")
        super().__init__(params, dict(lr=lr, betas=tuple(betas), eps=eps, weight_decay=weight_decay, amsgrad=False,
                                      maximize=maximize))
        self._tables = {}

    # state[p] = {'step', 'exp_avg', 'exp_avg_sq'} exactly like torch.optim.Adam; 'step' of every parameter of a
    # group is a view of the group's device step counter.
    def _group_state(self, group):
        ps = [p for p in group['params'] if p.grad is not None]
        if not ps:
            return ps, None
        ops._require_cuda(*ps)
        counter = group.get('_step_state')
        if counter is None or counter.device != ps[0].device:
            counter = torch.zeros(4, dtype=torch.float32, device=ps[0].device)
            # after load_state_dict (or a torch.optim.Adam state): continue from the restored count
            for p in group['params']:
                st = self.state.get(p)
                if st and 'step' in st:
                    counter[0] = float(st['step'])
                    break
            group['_step_state'] = counter
        for p in ps:
            if p.dtype != torch.float32 or not p.is_contiguous():
                raise _lib.CpcError("cpc_b200.optim.Adam needs contiguous fp32 parameters")
            st = self.state[p]
            if 'exp_avg' not in st:
                st['exp_avg'] = torch.zeros_like(p, memory_format=torch.contiguous_format)
                st['exp_avg_sq'] = torch.zeros_like(p, memory_format=torch.contiguous_format)
            st['step'] = counter[0]
        return ps, counter

    @torch.no_grad()
    def step(self, closure=None, flat_grads=None, grad_scale=1.0, skip_if=None):
        """``flat_grads``: optional {param: tensor} overriding ``p.grad`` as the gradient source (the all-reduced
        flat buffer of the multi-GPU step); ``grad_scale`` multiplies every gradient (1 / world size there).
        ``skip_if``: optional one-element fp32 tensor on the parameters' device, read by the kernels when they run; a
        non-zero value leaves parameters, moments and the step count untouched (``cpc_adam_step_ex``), so a step
        captured in a CUDA graph decides at each replay whether it applies."""
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        lib = _lib.load()
        for group in self.param_groups:
            ps, counter = self._group_state(group)
            if not ps:
                continue
            grads = [flat_grads[p] if flat_grads is not None else p.grad for p in ps]
            for g in grads:
                if g.dtype != torch.float32 or not g.is_contiguous() or g.is_sparse:
                    raise _lib.CpcError("cpc_b200.optim.Adam needs dense contiguous fp32 gradients")
            key = tuple((p.data_ptr(), g.data_ptr()) for p, g in zip(ps, grads))
            cached = self._tables.get(id(group))
            if cached is None or cached[0] != key:
                n = len(ps)
                arr = ctypes.c_void_p * n
                tables = (arr(*[p.data_ptr() for p in ps]), arr(*[g.data_ptr() for g in grads]),
                          arr(*[self.state[p]['exp_avg'].data_ptr() for p in ps]),
                          arr(*[self.state[p]['exp_avg_sq'].data_ptr() for p in ps]),
                          (ctypes.c_int64 * n)(*[p.numel() for p in ps]))
                cached = (key, tables)
                self._tables[id(group)] = cached
            t = cached[1]
            a = _lib.AdamParams(float(group['lr']), float(group['betas'][0]), float(group['betas'][1]),
                                float(group['eps']), float(group['weight_decay']), float(grad_scale),
                                int(bool(group['maximize'])))
            numel = float(sum(p.numel() for p in ps))
            if skip_if is not None and (skip_if.dtype != torch.float32 or skip_if.numel() != 1
                                        or skip_if.device != ps[0].device):
                raise _lib.CpcError("cpc_b200.optim.Adam: skip_if must be a one-element fp32 tensor on %s" % ps[0].device)
            with torch.cuda.device(ps[0].device):
                if skip_if is None:
                    ops._call("cpc_adam_step n%d" % len(ps), 0.0, lib.cpc_adam_step, len(ps), t[0], t[1], t[2], t[3],
                              t[4], ops._ptr(counter), ctypes.byref(a), ops._stream(), nbytes=28.0 * numel)
                else:
                    ops._call("cpc_adam_step_ex n%d" % len(ps), 0.0, lib.cpc_adam_step_ex, len(ps), t[0], t[1], t[2],
                              t[3], t[4], ops._ptr(counter), ops._ptr(skip_if), ctypes.byref(a), ops._stream(),
                              nbytes=28.0 * numel)
        return loss

    def state_dict(self):
        sd = super().state_dict()
        for g in sd['param_groups']:
            g.pop('_step_state', None)
        for st in sd['state'].values():
            if 'step' in st:
                st['step'] = st['step'].detach().clone()
        return sd

    def load_state_dict(self, state_dict):
        super().load_state_dict(state_dict)
        for group in self.param_groups:
            group.pop('_step_state', None)                     # rebuilt from the restored 'step' at the next step
        self._tables.clear()
