"""rough_rank DSSM (PLE user / item towers + cross-network teacher + distilled shallow student).

Reference: rough_rank/model.py (towers :16-86, embeddings :89-115, DSSM :118-187, losses :190-222) and
rough_rank/config/config.py (feature lists :77-83, `get_feature_id` :66-70).

    create_tower_teacher / create_tower / create_shallow_tower  -> nn.Modules with the reference's wiring
    DSSM()        -> {"train", "predict"}   (+ "net": the object with train_step)
    create_model()   dense Adam 1e-4, BCE(student) + BCE(teacher) + mean(distill)
"""
from __future__ import annotations

from typing import Dict, Optional, Sequence

import torch
from torch import nn

from .builders import _KerasDense
from .embedding import Adam, category_column, embedding_column
from .net import ComposedNet
from .rough_rank_layer import DNN, PLE, CrossNet, KDLoss


class config:
    """The resolved constants of rough_rank/config/config.py: in the shipped configuration every
    feature id equals its slot id (`FEATURE_ID` holds none of the 52 feature names, so
    `get_feature_id` falls through to `FEATURE_SLOT`, config.py:66-70)."""
    USER_FEATURE_IDS = ("2597 2 4 5 6 1567 1568 1570 1571 1572 1574 1575 1576 1577 1578 1579 1582 1586 1589 1736 2039 "
                        "2123 2125 2127 2128 2130 2131 2148 2150 2151 2153 2154 2155").split()            # :77-78
    ITEM_FEATURE_IDS = ("1591 1592 1593 1594 1595 1601 1614 1616 1624 1737 1738 2040 2041 2042 2043 2044 2045 2046 "
                        "2049").split()                                                                    # :80-81
    ALL_FEATURE_ID_2_SLOT = {f: int(f) for f in USER_FEATURE_IDS + ITEM_FEATURE_IDS}                       # :72
    ALL_FEATURE_SLOT = set(ALL_FEATURE_ID_2_SLOT.values())
    USER_OUTPUT_DIM = 16
    ITEM_OUTPUT_DIM = 16
    DENSE_MASK_ID = "4575"                                                                                # model.py:129

    @staticmethod
    def get_feature_id(feature_name):
        if str(feature_name) in config.ALL_FEATURE_ID_2_SLOT:
            return str(feature_name)
        raise ValueError("feature: {} not found".format(feature_name))


C = config


def dict_to_sorted_list(d, key_func=None):
    """model.py:10-13."""
    if key_func is None:
        key_func = lambda x: x[0]
    return [v for k, v in sorted(list(d.items()), key=key_func)]


class TeacherTower(nn.Module):
    """create_tower_teacher (model.py:16-34): CrossNet || Dense128-Dense64, concat, Dense16, Dense1 logit."""

    def __init__(self, tower_name="teacher"):
        super().__init__()
        self.tower_name = tower_name
        self.cross = CrossNet()
        self.dense0, self.dense1 = _KerasDense(128, "relu"), _KerasDense(64, "relu")
        self.dense2 = _KerasDense(16, None)
        self.pred = _KerasDense(1, None)                      # 'pred_<tower>'

    def forward(self, embs: Dict[str, torch.Tensor]):
        x = torch.cat(dict_to_sorted_list(embs), dim=-1)
        merge = torch.cat([self.dense1(self.dense0(x)), self.cross(x)], dim=-1)
        return {"logit": self.pred(self.dense2(merge))}


class Tower(nn.Module):
    """create_tower (model.py:37-67): PLE(4 shared + 4 specific experts of Dense(32)) -> DNN((output_dim,),
    linear) per task; with a mask tensor two tasks ('td', 'hpld') are built and selected per sample by
    `mask == 1` (:54-55)."""

    def __init__(self, tower_name, output_dim=16, with_mask=False):
        super().__init__()
        self.tower_name, self.with_mask = tower_name, with_mask
        nt = 2 if with_mask else 1
        self.ple = PLE(num_tasks=nt, num_shared_experts=4, num_specific_experts=4, expert_dnn_units=(32,),
                       gate_dnn_units=(), expert_dnn_params=dict(), gate_dnn_params=dict())
        self.heads = nn.ModuleList([DNN((output_dim,), output_activation="linear", l2_reg=0, dropout_rate=0)
                                    for _ in range(nt)])

    def forward(self, embs: Dict[str, torch.Tensor], mask_tensor: Optional[torch.Tensor] = None):
        x = torch.cat(dict_to_sorted_list(embs), dim=-1)
        ple = self.ple(x)
        outs = [h(p) for h, p in zip(self.heads, ple)]
        if self.with_mask:
            sel = (mask_tensor == 1).reshape(-1, 1)
            return {"emb": torch.where(sel, outs[1], outs[0])}
        return {"emb": outs[0]}


class ShallowTower(nn.Module):
    """create_shallow_tower (model.py:70-86): concat -> Dense(32, relu) -> Dense(1) logit -> sigmoid."""

    def __init__(self):
        super().__init__()
        self.shallow_dnn_0 = _KerasDense(32, "relu")
        self.logit_shallow = _KerasDense(1, None)

    def forward(self, deep_inputs: Sequence[torch.Tensor]):
        logit = self.logit_shallow(self.shallow_dnn_0(torch.cat(list(deep_inputs), dim=-1)))
        return {"logit": logit, "final_output": torch.sigmoid(logit)}


def create_tower_teacher(tower_name="teacher"):
    return TeacherTower(tower_name)


def create_tower(tower_name, output_dim=16, mask_tensor=None):
    return Tower(tower_name, output_dim, with_mask=mask_tensor is not None)


def create_shallow_tower():
    return ShallowTower()


class DssmSubModel(nn.Module):
    """The dense graph of DSSM() (model.py:130-170) on given embeddings."""

    def __init__(self, user_ids=C.USER_FEATURE_IDS, item_ids=C.ITEM_FEATURE_IDS):
        super().__init__()
        self.user_ids, self.item_ids = list(user_ids), list(item_ids)
        self.user = Tower("user", C.USER_OUTPUT_DIM, with_mask=True)
        self.item = Tower("item", C.ITEM_OUTPUT_DIM)
        self.teacher = TeacherTower("teacher")
        self.shallow = ShallowTower()
        self.distill = KDLoss()

    def forward(self, embs: Dict[str, torch.Tensor], dense_mask: torch.Tensor):
        user = self.user({f: embs[f] for f in self.user_ids}, dense_mask)["emb"]
        item = self.item({f: embs[f] for f in self.item_ids})["emb"]
        teacher_logit = self.teacher({f: embs[f] for f in self.user_ids + self.item_ids})["logit"]
        student = self.shallow([user, item])
        kd = self.distill(student["logit"], teacher_logit.detach())                    # :163-164
        return {"student": student["final_output"], "teacher": torch.sigmoid(teacher_logit), "distill": kd}


def mse_loss(y_true, y_pred):
    """model.py:190-198."""
    y = y_true.to(torch.float32) * 1.0 / 1000
    wt_log = torch.log(y + 1.0)
    return ((torch.clamp(wt_log, max=5.3) - y_pred) ** 2).mean()


def y_pred_loss(y_true, y_pred):
    return y_pred.mean()


def binary_crossentropy(y_true, y_pred, eps=1e-7):
    """tf.keras.losses.BinaryCrossentropy() on probabilities (clip to [eps, 1-eps], mean)."""
    p = y_pred.clamp(eps, 1.0 - eps)
    y = y_true.to(p.dtype)
    return (-(y * torch.log(p) + (1.0 - y) * torch.log(1.0 - p))).mean()


class DssmNet(ComposedNet):
    """DSSM() (model.py:118-187): 16-d embeddings (combiner mean, bucket 25600, sparse Adam 1e-3, :89-115)
    for the user and item feature ids + the dense mask input '4575'.  `train_step` is the create_model() compile
    (model.py:206-222): dense Adam 1e-4; BCE(student) + BCE(teacher) + mean(distill)."""
    dense_lr = 0.0001

    def __init__(self, user_ids=C.USER_FEATURE_IDS, item_ids=C.ITEM_FEATURE_IDS, bucket_size=25600,
                 device="cuda:0", seed=0, embedding_cls=None, group=None):
        self.ids = list(user_ids) + list(item_ids)
        dims = [C.USER_OUTPUT_DIM] * len(user_ids) + [C.ITEM_OUTPUT_DIM] * len(item_ids)
        cols = [embedding_column(category_column(C.get_feature_id(f) if f in C.ALL_FEATURE_ID_2_SLOT else f,
                                                 bucket_size), dimension=d, combiner="mean")
                for f, d in zip(self.ids, dims)]
        super().__init__(cols, Adam(learning_rate=0.001, beta1=0.9, beta2=0.999, epsilon=1e-8), "sparse_emb_input",
                         device, seed, embedding_cls, group)
        self.sub_model = DssmSubModel(user_ids, item_ids).to(device)

    def train(self, inputs):
        e = self.emb({k: v for k, v in inputs.items() if k != C.DENSE_MASK_ID})
        return self.sub_model(e, inputs[C.DENSE_MASK_ID].to(self.emb.dev))

    def predict(self, inputs):
        with torch.no_grad():
            return self.train(inputs)

    def _forward(self, x, inputs):
        return self.sub_model(x, inputs[C.DENSE_MASK_ID].to(self.emb.dev))

    def _loss(self, out, labels):
        return (binary_crossentropy(labels["student"], out["student"]) +
                binary_crossentropy(labels["teacher"], out["teacher"]) + y_pred_loss(None, out["distill"]))


def DSSM(**kw):
    net = DssmNet(**kw)
    return {"train": net.train, "predict": net.predict, "net": net}


def create_model(**kw):
    return DSSM(**kw)
