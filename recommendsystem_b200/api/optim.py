"""Dense-parameter optimizer of the composed models: `tn.optimizer.Optimizer(tn.core.Adam(...))`
(rank/multi_head/model.py:52-53, staytime/model.py:75, rough_rank/model.py:209, rank/ctr/base_model.py:192).

All trainable parameters of a sub-model are re-homed into ONE flat fp32 buffer (each nn.Parameter becomes a
16-byte-aligned view of it, its .grad a view of a flat gradient buffer), so that a step is two launches whatever
the number of layers: rs_adam_advance (step counter and bias corrections on the device: CUDA-graph replays advance
the optimizer) + rs_dense_adam.  Multi-GPU data parallelism all-reduces the flat gradient buffer once.
"""
from __future__ import annotations

from typing import Iterable

import torch

from .. import ops


class DenseAdam:
    def __init__(self, params: Iterable[torch.nn.Parameter], lr, beta1=0.9, beta2=0.999, eps=1e-8, group=None):
        self.params = [p for p in params if p.requires_grad]
        if not self.params:
            raise ValueError("DenseAdam: no trainable parameters (build the lazily-built layers with one forward first)")
        dev = self.params[0].device
        if dev.type != "cuda":
            raise RuntimeError("DenseAdam runs on CUDA tensors only (no CPU fallback)")
        self.lr, self.beta1, self.beta2, self.eps = float(lr), float(beta1), float(beta2), float(eps)
        offs, n = [], 0
        for p in self.params:
            offs.append(n)
            n += (p.numel() + 3) // 4 * 4
        self.flat = torch.zeros(n, device=dev)
        self.flat_g = torch.zeros(n, device=dev)
        self.flat_m = torch.zeros(n, device=dev)
        self.flat_v = torch.zeros(n, device=dev)
        self.scalars = torch.zeros(4, device=dev)
        with torch.no_grad():
            for p, o in zip(self.params, offs):
                if p.dtype != torch.float32:
                    raise TypeError("DenseAdam: fp32 master parameters")
                view = self.flat[o:o + p.numel()].view(p.shape)
                view.copy_(p.data)
                p.data = view
                p.grad = self.flat_g[o:o + p.numel()].view(p.shape)
        self.offsets = offs
        self.group = group            # torch.distributed group: gradients are averaged over its ranks

    def zero_grad(self):
        """Gradients accumulate into the flat buffer's views (autograd adds in place): one memset clears them."""
        self.flat_g.zero_()

    def step(self):
        if self.group is not None:
            import torch.distributed as dist
            if dist.get_world_size(self.group) > 1:
                if dist.get_backend(self.group) == "nccl":
                    dist.all_reduce(self.flat_g, op=dist.ReduceOp.AVG, group=self.group)
                else:
                    dist.all_reduce(self.flat_g, group=self.group)
                    self.flat_g.div_(dist.get_world_size(self.group))
        ops.adam_advance(self.scalars, self.beta1, self.beta2)
        ops.dense_adam(self.flat, self.flat_m, self.flat_v, self.flat_g, self.lr, self.beta1, self.beta2, self.eps,
                       self.scalars, None)

    def moments(self):
        """(parameter, m, v) of every parameter: views of the flat moment buffers shaped like the parameter."""
        for p, o in zip(self.params, self.offsets):
            k = p.numel()
            yield p, self.flat_m[o:o + k].view(p.shape), self.flat_v[o:o + k].view(p.shape)

    # state that one step changes (GraphedTrainStep undoes its warm-up with these)
    def snapshot(self):
        return [t.clone() for t in (self.flat, self.flat_m, self.flat_v, self.scalars)]

    def restore(self, snap):
        for t, s in zip((self.flat, self.flat_m, self.flat_v, self.scalars), snap):
            t.copy_(s)
