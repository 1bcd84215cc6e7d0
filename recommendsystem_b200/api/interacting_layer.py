"""InteractingLayer — drop-in for the reference's Keras layer (InteractingLayer.py:7-61, duplicated
at rank/multi_head/interacting_layer.py): multi-head self-attention over the feature fields with
ReLU Dense projections, residual, ReLU and LayerNorm, the SAME weights re-applied `layer_num` times."""
from __future__ import annotations

import math

import torch
from torch import nn

from .functional import InteractingFn


class InteractingLayer(nn.Module):
    """InteractingLayer(layer_num=1, unit_num=128, head_num=1, use_dropout=False, dropout_rate=0.3,
    use_res=True) — the reference signature (InteractingLayer.py:9-16).  `unit_num` is the TOTAL width
    (per head: unit_num // head_num, :47-51).

    Extra keyword `ln_eps` pins the epsilon of the LayerNormalization whose source is missing from
    the reference (InteractingLayer.py:4); default 1e-3 = tf.keras.layers.LayerNormalization.
    `use_dropout=True` applies inverted dropout to the attention weights in training mode (:53-54) inside the
    fused kernels (counter-based mask, seed `dropout_seed` + call counter; TF's own random stream cannot be
    reproduced, the distribution can).
    Weights are created on the first call (Keras `build`), Keras layout and names:
    query_dense/key_dense/value_dense/res_dense .kernel [in, unit_num] and .bias, layer_norm.gamma/.beta.
    """

    def __init__(self, layer_num=1, unit_num=128, head_num=1, use_dropout=False, dropout_rate=0.3,
                 use_res=True, ln_eps=1e-3, **kwargs):
        super().__init__()
        self.layer_num, self.unit_num, self.head_num = int(layer_num), int(unit_num), int(head_num)
        self.use_dropout, self.dropout_rate, self.use_res = bool(use_dropout), float(dropout_rate), bool(use_res)
        self.ln_eps = float(ln_eps)
        self.dropout_seed = int(kwargs.get("dropout_seed", 0x5DEECE66D))     # masks = f(seed, call counter)
        self._dropout_calls = 0
        self._drop_step = None               # device-side call counter (int64[1]), created at the first training call
        self.last_dropout_seed = None
        if self.unit_num % self.head_num != 0:
            raise ValueError("head_num must divide unit_num (tf.split, InteractingLayer.py:47)")
        self.built = False

    @classmethod
    def from_deepctr(cls, att_embedding_size, head_num=2, use_res=True, **kw):
        """DeepCTR-style alias named by BASELINE.json: att_embedding_size is PER HEAD, one iteration."""
        return cls(layer_num=1, unit_num=att_embedding_size * head_num, head_num=head_num, use_res=use_res, **kw)

    def build(self, input_shape, device=None, dtype=torch.float32):
        if len(input_shape) != 3:
            raise ValueError('The rank of input of InteractingLayer must be 3, but now is %d' % len(input_shape))
        D, U = int(input_shape[-1]), self.unit_num
        if self.layer_num > 1 and D != U:
            raise ValueError("layer_num > 1 re-applies the Dense layers to their own output: input dim must "
                             "equal unit_num (InteractingLayer.py:41-46)")
        lim = math.sqrt(6.0 / (D + U))              # Keras Dense default: glorot_uniform kernel, zero bias
        for name in ("query_dense", "key_dense", "value_dense", "res_dense"):
            self.register_parameter(name + "_kernel", nn.Parameter(torch.empty(D, U, device=device).uniform_(-lim, lim)))
            self.register_parameter(name + "_bias", nn.Parameter(torch.zeros(U, device=device)))
        self.layer_norm_gamma = nn.Parameter(torch.ones(U, device=device))
        self.layer_norm_beta = nn.Parameter(torch.zeros(U, device=device))
        self.built = True

    def packed(self):
        W = torch.cat([self.query_dense_kernel, self.key_dense_kernel, self.value_dense_kernel,
                       self.res_dense_kernel], dim=1)
        b = torch.cat([self.query_dense_bias, self.key_dense_bias, self.value_dense_bias, self.res_dense_bias])
        return W, b

    def forward(self, inputs):
        if inputs.dim() != 3:
            raise ValueError('The rank of input of InteractingLayer must be 3, but now is %d' % inputs.dim())
        if not self.built:
            self.build(inputs.shape, device=inputs.device)
        rate, seed, step = 0.0, 0, None
        if self.use_dropout and self.training:
            # tf.keras Dropout on the attention weights (InteractingLayer.py:53-54): a fresh counter-based mask per
            # call.  The call counter lives on the DEVICE and is bumped in-stream: a CUDA graph of the step (api.graph)
            # advances it on every replay, so replays draw fresh masks (a host-side counter would be frozen into the
            # graph).  Effective seed of call k (1-based) = dropout_seed + 0x9E3779B97F4A7C15 * k.
            rate = float(self.dropout_rate)
            seed = self.dropout_seed & 0xFFFFFFFFFFFFFFFF
            if self._drop_step is None or self._drop_step.device != inputs.device:
                self._drop_step = torch.zeros(1, dtype=torch.int64, device=inputs.device)
            self._drop_step.add_(1)
            step = self._drop_step
            self._dropout_calls += 1            # host mirror (valid while the layer runs eagerly)
            self.last_dropout_seed = (seed + 0x9E3779B97F4A7C15 * self._dropout_calls) & 0xFFFFFFFFFFFFFFFF
        W, b = self.packed()
        return InteractingFn.apply(inputs, W, b, self.layer_norm_gamma, self.layer_norm_beta, self.ln_eps,
                                   self.head_num, self.layer_num, self.use_res, rate, seed, step)

    def dropout_state(self):
        """(host call count, device call count) of the dropout mask counter: the state a training call advances."""
        return self._dropout_calls, 0 if self._drop_step is None else int(self._drop_step.item())

    def load_dropout_state(self, state):
        """Set the counter to a dropout_state() value, in place: a captured CUDA graph of the step keeps reading it."""
        self._dropout_calls, step = (int(x) for x in state)
        if self._drop_step is not None:
            self._drop_step.fill_(step)
        elif step:
            self._drop_step = torch.full((1,), step, dtype=torch.int64, device=self.layer_norm_gamma.device)

    def get_config(self):
        return dict(layer_num=self.layer_num, unit_num=self.unit_num, head_num=self.head_num,
                    use_dropout=self.use_dropout, dropout_rate=self.dropout_rate, use_res=self.use_res,
                    ln_eps=self.ln_eps)


def dropout_layers(module: nn.Module):
    """(path, layer) of every InteractingLayer in `module`: the layers whose dropout counter a train step advances."""
    return [(p, m) for p, m in module.named_modules() if isinstance(m, InteractingLayer)]
