"""Model builders of the reference's CTR path, wired from the drop-in layers.

    AutoInt(model_config).run()                     autoint:11-60 (+ rank/ctr/base_model.py output_layer)
    AUTOINT(linear_features, dense_features, training, dnn_hidden_units) -> ModelResult
                                                    rank/multi_head/multidnn.py:14-259 (AutoInt + DNN +
                                                    7-expert / 7-gate MMoE, 7 sigmoid heads)
    cross_entropy                                   rank/multi_head/model.py:18-22, rank/ctr/base_model.py:7-12

AutoInt is backed by the captured single-launch-stream engine (recommendsystem_b200.autoint); AUTOINT
is an nn.Module over the autograd wrappers (every Dense / InteractingLayer forward+backward is a C-ABI
kernel) whose sparse side is api.embedding.EmbeddingFeatures.
"""
from __future__ import annotations

from typing import Dict, Sequence

import torch
from torch import nn

from ..autoint import AutoIntConfig, AutoIntTrainer
from .embedding import Adam, EmbeddingFeatures, category_column, embedding_column
from .optim import DenseAdam
from .functional import dense
from .interacting_layer import InteractingLayer


def cross_entropy(y_true, y_pred, a=1.0, reduce_mean=False):
    """-y log(p+1e-6) - (a-y) log(1-p+1e-6), summed over the label axis (keepdims);
    rank/multi_head/model.py:18-22.  reduce_mean=True: mean over the batch (rank/ctr/base_model.py:7-12)."""
    l = -y_true * torch.log(y_pred + 1e-6) - (a - y_true) * torch.log(1 - y_pred + 1e-6)
    l = l.sum(dim=1, keepdim=True)
    return l.mean() if reduce_mean else l


class AutoInt:
    """AutoInt(model_config) — autoint:11-60.  model_config['model_param'] follows the keys the reference
    reads (:30-41,49-50): interact{layer_num,unit_num,head_num,use_dropout,dropout_rate,use_res},
    mlp{hidden_units,activation}, logits{hidden_units,activation}; plus 'feature' {num_fields,
    rows_per_field, embed_dim} and optional 'batch', 'dtype', 'ln_eps' for the synthetic setting (the
    reference's JSON slot bookkeeping, rank/ctr/base_model.py:35-158, is a "next" row in SURVEY §8f)."""

    def __init__(self, model_config: Dict, device="cuda:0", **kwargs):
        self.model_config = model_config
        mp, ft = model_config["model_param"], model_config["feature"]
        it = mp["interact"]
        if mp["mlp"].get("activation", "relu") != "relu":
            raise NotImplementedError("the fused AutoInt engine implements the relu tower")
        lg = mp.get("logits", {"hidden_units": [1], "activation": "sigmoid"})
        if list(lg["hidden_units"]) != [1] or lg["activation"] != "sigmoid":
            raise NotImplementedError("logits head: Dense(1, sigmoid) (autoint:49-52 clips to a probability)")
        if it.get("use_dropout", False):
            raise NotImplementedError("the captured AutoInt engine runs without attention dropout; use "
                                      "api.InteractingLayer(use_dropout=True) in a module graph")
        self.cfg = AutoIntConfig(num_fields=ft["num_fields"], rows_per_field=ft["rows_per_field"],
                                 embed_dim=ft["embed_dim"], layer_num=it["layer_num"], unit_num=it["unit_num"],
                                 head_num=it["head_num"], use_res=it.get("use_res", True),
                                 ln_eps=model_config.get("ln_eps", 1e-3), mlp_hidden=tuple(mp["mlp"]["hidden_units"]),
                                 batch=model_config.get("batch", 8192), dtype=model_config.get("dtype", "f32"))
        self.device = device

    def run(self):
        trainer = AutoIntTrainer(self.cfg, self.device)
        return {"train": trainer, "predict": trainer.predict}


class _KerasDense(nn.Module):
    def __init__(self, units, activation=None, init_std=None):
        super().__init__()
        self.units, self.activation, self.init_std = units, activation, init_std
        self.kernel = None

    def forward(self, x):
        if self.kernel is None:
            fan_in = x.shape[-1]
            w = torch.empty(fan_in, self.units, device=x.device)
            if self.init_std is None:
                lim = (6.0 / (fan_in + self.units)) ** 0.5
                w.uniform_(-lim, lim)
            else:
                nn.init.trunc_normal_(w, std=self.init_std, a=-2 * self.init_std, b=2 * self.init_std)
            self.kernel = nn.Parameter(w)
            self.bias = nn.Parameter(torch.zeros(self.units, device=x.device))
        return dense(x, self.kernel, self.bias, self.activation)


def fused_dense(x, layers, activation):
    """Dense layers of the reference that read the SAME input (the per-expert / per-gate first layers of the MMoE blocks,
    staytime/VideoDnn.py:130-164, rank/multi_head/multidnn.py:80-99) evaluated as ONE GEMM over their kernels laid side by
    side — x is read once, the input gradient is one dgrad GEMM instead of one per layer plus their sum.  The layers keep
    their own parameters (Keras names, state_dict keys); returns [.., sum(units)], split it with `[l.units for l in layers]`."""
    for l in layers:
        if l.kernel is None:
            l(x[:1])                                  # first call: creates kernel / bias exactly as the layer itself would
    return dense(x, torch.cat([l.kernel for l in layers], dim=1), torch.cat([l.bias for l in layers]), activation)


# rank/multi_head/multidnn.py:206-209 MultiLabelInfo.label_list: the names (and order) of the 7 outputs
AUTOINT_LABELS = ["like_pred", "click_comment_pred", "comment_pred", "click_sharing_pred", "follow_pred",
                  "click_avatar_pred", "unlike_pred"]


class AutoIntSubModel(nn.Module):
    """create_autoint_sub_model (rank/multi_head/multidnn.py:14-212): InteractingLayer(1, 8, 2 heads, dropout 0.2) ||
    Dense stack dnn_{i} -> concat -> experts expert_{i}_fc1 Dense(32, relu) (8 built, the first 7 used, :80-92) ->
    7 softmax gates gate_{i}_fc2 -> 7 sigmoid heads named like the labels.  Sub-modules carry the reference's Keras
    layer names, so `state_dict()` keys are `<keras name>.kernel / .bias` and `interacting_layer.*`."""

    NUM_LABELS = 7

    def __init__(self, deep_hidden_units: Sequence[int] = (32, 16), expert_num=7, expert_units=32):
        super().__init__()
        # multidnn.py:54: attention dropout 0.2 in training (fused into the kernel, counter-based mask)
        self.interacting_layer = InteractingLayer(layer_num=1, unit_num=8, head_num=2, use_dropout=True,
                                                  dropout_rate=0.2, use_res=True)
        for i, u in enumerate(deep_hidden_units):
            self.add_module("dnn_%d" % i, _KerasDense(u, "relu"))
        for i in range(expert_num + 1):
            self.add_module("expert_%d_fc1" % i, _KerasDense(expert_units, "relu", 0.001))
        for i in range(self.NUM_LABELS):
            self.add_module("gate_%d_fc2" % i, _KerasDense(expert_num, "softmax", 0.001))
        for label in AUTOINT_LABELS:
            self.add_module(label, _KerasDense(1, "sigmoid"))
        self.n_deep, self.expert_num = len(deep_hidden_units), expert_num

    def forward(self, embs: Sequence[torch.Tensor]):
        all_inputs = torch.stack(list(embs), dim=1)                       # :25-27,50  [B,F,8]
        autoint = self.interacting_layer(all_inputs).flatten(1)           # :54-56
        deep = all_inputs.flatten(1)                                      # :60
        for i in range(self.n_deep):
            deep = getattr(self, "dnn_%d" % i)(deep)                      # :62-63
        result = torch.cat([deep, autoint], dim=1)                        # :72
        # every expert is evaluated as the reference builds it; only [0:7] feed the gates (:92).  The 8 experts
        # (Dense(32, relu)) and the 7 gates (Dense(7, softmax)) all read `result`: one GEMM each group
        B, E, L = result.shape[0], self.expert_num, self.NUM_LABELS
        ex_layers = [getattr(self, "expert_%d_fc1" % i) for i in range(E + 1)]
        experts = fused_dense(result, ex_layers, "relu").view(B, E + 1, ex_layers[0].units)[:, :E]       # [B,7,32]
        gates = fused_dense(result, [getattr(self, "gate_%d_fc2" % i) for i in range(L)], None)
        gates = torch.softmax(gates.view(B, L, E), dim=-1)                                              # :97-99
        mixed = (experts.unsqueeze(1) * gates.unsqueeze(-1)).sum(dim=2)                                  # :104-108 [B,L,32]
        # the 7 sigmoid heads Dense(1) (:118-206): pred_l = sigmoid(mixed_l . w_l + b_l)
        heads = [getattr(self, label) for label in AUTOINT_LABELS]
        for l, h in enumerate(heads):
            if h.kernel is None:
                h(mixed[:1, l])
        Wh = torch.stack([h.kernel[:, 0] for h in heads], dim=0)                                         # [L,32]
        bh = torch.cat([h.bias for h in heads])
        return torch.sigmoid((mixed * Wh.unsqueeze(0)).sum(dim=-1) + bh)  # [B,7] in label_list order


class ModelResult:
    """src.pipeline.model_result.ModelResult (not vendored by the reference; rank/multi_head/multidnn.py:247-250
    fills `model`, `sub_model`, `model_predict`)."""
    model = None
    sub_model = None
    model_predict = None


class _AutoIntFullModel:
    """`full_model` of AUTOINT: sparse ids -> EmbeddingFeatures -> sub_model.  Callable like a Keras model
    (`model(inputs)` -> [B,7] predictions); train_step() runs forward, the summed 7-label BCE
    (rank/multi_head/model.py:18-22), backward, the dense Adam (lr 1e-5, :52-53: rs_dense_adam) and the sparse push."""

    def __init__(self, slots, emb, sub_model, training, group=None):
        self.slots, self.emb, self.sub_model, self.training = slots, emb, sub_model, bool(training)
        self.opt = None
        self.group = group
        self.sub_model.train(self.training)

    def __call__(self, inputs: Dict[str, torch.Tensor]):
        return self.predict(inputs)

    def predict(self, inputs: Dict[str, torch.Tensor]):
        was = self.sub_model.training
        self.sub_model.eval()
        try:
            with torch.no_grad():
                embs = self.emb(inputs)
                return self.sub_model([embs[s] for s in self.slots])
        finally:
            self.sub_model.train(was)

    def train_step(self, inputs: Dict[str, torch.Tensor], labels):
        if isinstance(labels, dict):
            labels = torch.cat([labels[k].reshape(-1, 1) for k in AUTOINT_LABELS], dim=1)
        embs = self.emb(inputs)
        leaves = [embs[s].detach().requires_grad_(True) for s in self.slots]
        pred = self.sub_model(leaves)
        opt = self.dense_optimizer()
        loss = cross_entropy(labels, pred).mean()
        opt.zero_grad()
        loss.backward()
        opt.step()
        self.emb.backward({s: l.grad for s, l in zip(self.slots, leaves)})
        return loss.detach(), pred.detach()

    def dense_optimizer(self):
        """The dense Adam of sub_model (lr 1e-5), created at the first call: the lazily-built layers must exist."""
        if self.opt is None:
            self.opt = DenseAdam(self.sub_model.parameters(), lr=1e-5, beta1=0.9, beta2=0.999, eps=1e-8, group=self.group)
        return self.opt

    # the InteractingLayer's device-side dropout counter is part of what a step changes (api.graph warm-up undo)
    def extra_state_snapshot(self):
        il = self.sub_model.interacting_layer
        return (il._dropout_calls, None if il._drop_step is None else il._drop_step.clone())

    def extra_state_restore(self, st):
        il = self.sub_model.interacting_layer
        il._dropout_calls = st[0]
        if il._drop_step is not None:
            if st[1] is None:
                il._drop_step.zero_()
            else:
                il._drop_step.copy_(st[1])


def create_autoint_sub_model(slot_zip_user_embs, dense_inputs_map, deep_hidden_units, training, device="cuda:0"):
    """rank/multi_head/multidnn.py:14.  `slot_zip_user_embs` (slot, embedding) pairs fix the input order; the
    `dense_inputs_map` inputs are declared by the reference but feed nothing (:30-31 vs :211)."""
    del slot_zip_user_embs, dense_inputs_map
    return AutoIntSubModel(deep_hidden_units).to(device).train(bool(training))


def AUTOINT(linear_features, dense_features, training, dnn_hidden_units=(32, 16), *, bucket_size=100_000,
            device="cuda:0", seed=0, embedding_cls=None, group=None, id_map="mod"):
    """AUTOINT(linear_features, dense_features, training, dnn_hidden_units=(32,16)) -> ModelResult{model, sub_model,
    model_predict} — rank/multi_head/multidnn.py:214-259.  8-d embeddings (combiner mean, tn.core.Adam lr 5e-5,
    :222,235) of the sorted, de-duplicated slots (:215-218) feed create_autoint_sub_model in `linear_features` order
    (:239).  Keyword-only extras stand in for the missing `src.*` Config: bucket_size (rows per slot table), device,
    seed; embedding_cls / group select the row-sharded multi-GPU embedding (api.sharded_embedding); id_map="hash" gives
    every distinct slot id its own row (api.embedding.EmbeddingFeatures)."""
    features = sorted(set(linear_features))                                   # :215-218
    cols = [embedding_column(category_column(s, bucket_size), dimension=8, combiner="mean") for s in features]
    E = embedding_cls or EmbeddingFeatures
    kw = {"group": group} if embedding_cls is not None else {}      # None = the default process group
    if id_map != "mod":
        kw["id_map"] = id_map
    emb = E(cols, Adam(5e-5, 0.9, 0.999, 1e-8), "linear", device=device, seed=seed, **kw)
    sub_model = create_autoint_sub_model([(s, None) for s in linear_features], {k: None for k in dense_features},
                                         dnn_hidden_units, training, device=device)
    if embedding_cls is not None and group is None:
        from .optim import _world_group
        group = _world_group()
    full = _AutoIntFullModel(list(linear_features), emb, sub_model, training, group=group)
    ret = ModelResult()
    ret.model = full                                                           # :247
    ret.sub_model = sub_model                                                  # :248
    ret.model_predict = full.predict                                           # :249
    return ret
