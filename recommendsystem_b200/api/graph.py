"""Whole-step CUDA graphs for the composed models (VideoDnn MTL, DSSM, rank/ctr, AUTOINT).

The models' train steps are hundreds to a thousand small launches (one Dense / gate / slice per reference
layer) driven from Python autograd: on a B200 the step is bound by the host, not by the GPU.  Every launch in
them is capture-safe (the C-ABI kernels run on the current stream with caller-owned memory, the dense optimizer
is `capturable`, no host read-back), so the whole step - embedding gather, forward, backward, dense Adam, key
sort + sorted-segment sparse update - is captured ONCE and replayed:

    step = GraphedTrainStep(net, example_inputs, example_labels)      # warm-up + capture
    loss, outputs = step(inputs, labels)                               # copy into the static buffers, replay

The warm-up steps (they allocate workspaces) are UNDONE before the capture: the embedding rows they touched, the dense
parameters, both optimizers' state and the InteractingLayers' dropout counters are restored bit for bit, so capturing
after loading a checkpoint does not change the loaded weights and the first replay is the first train step.

`net` is a composed net (api.net: `emb`, `sub_model`, `opt` / `dense_optimizer()`, `predict`, `train_step(inputs: dict,
labels: dict) -> (loss, outputs)`), e.g. api.video_dnn.MtlNet, api.rough_rank_model.DssmNet, api.rank_ctr.RankCtrNet,
the AUTOINT model.  Shapes and dtypes are fixed by the example batch;
a different batch size needs its own GraphedTrainStep.  Inputs may live on the host (pinned or not): the copy
into the static device buffers is the only per-step host work besides the replay.
"""
from __future__ import annotations

from typing import Dict

import torch

from .interacting_layer import dropout_layers


def _static(d: Dict, dev):
    out = {}
    for k, v in d.items():
        out[k] = v.to(dev).clone() if isinstance(v, torch.Tensor) else v
    return out


class GraphedTrainStep:
    def __init__(self, net, inputs: Dict, labels: Dict, device=None, warmup: int = 3):
        dev = torch.device(device) if device is not None else next(
            v.device for v in list(labels.values()) + list(inputs.values()) if isinstance(v, torch.Tensor) and v.is_cuda)
        if dev.type != "cuda":
            raise RuntimeError("GraphedTrainStep needs a CUDA device")
        self.net, self.dev = net, dev
        self.inputs, self.labels = _static(inputs, dev), _static(labels, dev)
        snap = self._snapshot(net, self.inputs)
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            for _ in range(max(1, warmup)):          # allocates workspaces
                net.train_step(self.inputs, self.labels)
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        self._restore(net, snap)
        torch.cuda.synchronize(dev)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.loss, self.outputs = net.train_step(self.inputs, self.labels)
        self.warmup_steps = 0                        # the warm-up steps were undone: replay 1 is train step 1

    @staticmethod
    def _snapshot(net, inputs):
        """Everything the warm-up steps change.  The lazily built layers are built first and the dense optimizer is
        created, so that there are initial weights and optimizer state to return to.  The dropout counters are taken
        before that forward: a sub_model in training mode advances them in `predict` too."""
        dropout = [(m, m.dropout_state()) for _, m in dropout_layers(net.sub_model)]
        with torch.no_grad():
            net.predict(inputs)
        opt = net.dense_optimizer()
        return {"emb": net.emb.snapshot(inputs), "params": [p.detach().clone() for p in net.sub_model.parameters()],
                "opt": opt.snapshot(), "dropout": dropout}

    @staticmethod
    def _restore(net, snap):
        net.emb.restore(snap["emb"])
        net.opt.restore(snap["opt"])
        with torch.no_grad():
            for p, v in zip(net.sub_model.parameters(), snap["params"]):
                p.copy_(v)
        for layer, state in snap["dropout"]:
            layer.load_dropout_state(state)

    def __call__(self, inputs: Dict, labels: Dict):
        for k, v in inputs.items():
            if isinstance(v, torch.Tensor):
                self.inputs[k].copy_(v, non_blocking=True)
        for k, v in labels.items():
            if isinstance(v, torch.Tensor):
                self.labels[k].copy_(v, non_blocking=True)
        self.graph.replay()
        return self.loss, self.outputs
