"""staytime VideoDnn multi-task model (reference: staytime/VideoDnn.py, staytime/model.py).

    create_moe_sub_model(...)   -> VideoDnnSubModel     dense graph, staytime/VideoDnn.py:27-215
    mtl_net(slots, seq_slots, seq_max_len, dnn_hidden_units) -> {"train", "predict"}     :266-302
    create_model_func()                                  staytime/model.py:68-92
    custom_kl_loss / cross_entropy / mse_loss / huber_loss   staytime/model.py:20-60

Every Dense is `functional.dense` (C-ABI GEMM forward + backward), the three DIN units are the fused
DIN-B kernel reading `seq[:, :, 0:16]` in place, the sparse side is `EmbeddingFeatures` (gather +
sorted-segment AdaGrad).  Concats / gating products / softmax are torch CUDA glue.  Layer names follow
the reference's Keras layer names so that weights can be exchanged by name.
"""
from __future__ import annotations

from typing import Dict, Sequence

import torch
from torch import nn

from .builders import _KerasDense, fused_dense
from .embedding import AdaGrad, category_column, embedding_column
from .net import ComposedNet
from .staytime_config import Config as C
from .staytime_layer import DIN, DeepCrossLayer

USER_SLOTS = ["1568", "1589", "2039", "1570"]                         # VideoDnn.py:32
ITEM_SLOTS = ["1591", "1593", "1737", "1614"]                         # :33
BIAS_SLOTS = ["3051", "1570", "2039", "2544", "1568", "3376", "3365", "3369", "2597", "1737", "1593", "1591",
              "1589", "1614"]                                         # :34-35
DIN_QUERY = {"2125": "1591", "2128": "1593"}                          # :72-77 (anything else -> l1 cate 1737)
FFM_SLOTS = [[USER_SLOTS, ITEM_SLOTS, 8]]                             # :117


def _name(task):
    return "%s_%s" % (C.model_name, task.replace("_pred", ""))


TASK_KEYS = [_name(t) for t in C.task_names]                          # ..._staytime, ..._shortplay, ..._longplay


class VideoDnnSubModel(nn.Module):
    """create_moe_sub_model (staytime/VideoDnn.py:27-215).

    forward(embs, seqs) with `embs`: dict slot -> [B,32] and `seqs`: dict seq slot -> ([B,T,32], mask [B,T]);
    slots are visited in sorted order (mtl_net :282,296).  Returns (train_outputs, predict_outputs)."""

    def __init__(self, slots: Sequence[str], seq_slots: Sequence[str], deep_hidden_units=(256, 128)):
        super().__init__()
        self.slots = sorted(slots)
        self.seq_slots = sorted(seq_slots)
        self.units = tuple(deep_hidden_units)
        n = len(self.slots)
        D = _KerasDense
        self.din = nn.ModuleDict({"din_%s" % s: DIN() for s in self.seq_slots})                       # :76
        self.senet_squeeze_layer1 = D(int(n / 4), "relu")                                             # :82,88
        self.senet_extract_layer2 = D(n, "sigmoid")                                                   # :83,91
        self.ffm = nn.ModuleDict()
        for xs, ys, dim in FFM_SLOTS:                                                                 # :11-25
            for x in xs:
                for y in ys:
                    self.ffm["ffm_x_%s_%s_%d" % (x, y, dim)] = D(dim, None)
                    self.ffm["ffm_y_%s_%s_%d" % (x, y, dim)] = D(dim, None)
        self.experts = nn.ModuleDict()
        for i in range(C.num_experts):                                                                # :130-148
            for j, unit in enumerate(self.units):
                self.experts["gate_%d_%d_1" % (i, j)] = D(unit, "relu")
                self.experts["gate_%d_%d_2" % (i, j)] = D(unit, "sigmoid")
                self.experts["expert_output_%d_%d" % (i, j)] = D(unit, "relu")
        self.task_gates = nn.ModuleDict()
        for i in range(C.num_tasks):                                                                  # :153-164
            for j, unit in enumerate([64, 32]):
                self.task_gates["gate_%d_%d" % (i, j)] = D(unit, "relu")
            self.task_gates["gate_output_%d" % i] = D(C.num_experts, "softmax")
        self.cross = DeepCrossLayer(num_layer=3)                                                      # :167
        self.staytime_output = D(C.multiclass_num, None)                                              # :169
        self.tower_deep = nn.ModuleDict({"tower_deep_%s" % t: D(1, "relu") for t in C.task_names[1:]})  # :181,187
        self.tower_out = nn.ModuleDict({t: D(1, "sigmoid") for t in C.task_names[1:]})                # :184,190
        self.register_buffer("wt_bins", torch.tensor(C.bin_list, dtype=torch.float32).view(C.multiclass_num, 1))

    def _slot_indices(self, pos, bias_idx, device):
        """Index tensors of the user / item / bias slots on `device`, created once (a host->device copy is not
        capturable in a CUDA graph)."""
        cache = self.__dict__.setdefault("_idx_cache", {})
        if device not in cache:
            cache[device] = (torch.as_tensor([pos[s] for s in USER_SLOTS], device=device),
                             torch.as_tensor([pos[s] for s in ITEM_SLOTS], device=device),
                             torch.as_tensor(bias_idx, device=device))
        return cache[device]

    def forward(self, embs, seqs: Dict[str, tuple]):
        """embs: dict slot -> [B,32], or ONE stacked tensor [B, n, 32] whose slot axis is in sorted-slot order (what
        MtlNet hands over: the embedding layer's gather output as it lies).  Every per-slot step of the reference
        (slicing :45-48, SENet re-weighting :94-96, FM :107-115) is evaluated on the stacked tensor — one launch
        instead of one per slot."""
        G = torch.stack([embs[s] for s in self.slots], dim=1) if isinstance(embs, dict) else embs    # [B, n, 32]
        B, n = G.shape[0], G.shape[1]
        pos = {s: i for i, s in enumerate(self.slots)}
        general = G[:, :, 0:16]                                                                       # :47-48
        bias_idx = [pos[s] for s in self.slots if s in BIAS_SLOTS]                                    # :45-46
        din_embs = []
        for s in self.seq_slots:                                                                      # :53-77
            seq, mask = seqs[s]
            query = general[:, pos[DIN_QUERY.get(s, "1737")], :]
            din_embs.append(self.din["din_%s" % s](query.contiguous(), seq[:, :, 0:16], mask))
        # SENet re-weighting on a stop-gradient copy (:80-96)
        squeeze = general.reshape(B, n * 16).detach()
        w = 2.0 * self.senet_extract_layer2(self.senet_squeeze_layer1(squeeze))                       # [B, n]
        reweight = general * w.unsqueeze(-1)                                                          # [B, n, 16]
        # user x item products (:98-105), un-reweighted embeddings
        uidx, iidx, bidx = self._slot_indices(pos, bias_idx, G.device)
        mult = torch.relu(general.index_select(1, uidx).reshape(B, -1) * general.index_select(1, iidx).reshape(B, -1))
        # FM second-order term over the re-weighted embeddings (:107-115)
        sum_embs = reweight.sum(1)
        cross_term = sum_embs * sum_embs - (reweight * reweight).sum(1)
        fm_logit = 0.5 * cross_term.sum(-1, keepdim=True)
        # FFM (:117-120, 11-25)
        # (the |ys| projections of one user slot read the same 16 columns, and so do the |xs| projections of one item slot:
        # one GEMM per slot instead of one per pair, then ONE product over the [x, y, dim] grid)
        ffm = []
        for xs, ys, dim in FFM_SLOTS:
            gx = [general[:, pos[x], :].contiguous() for x in xs]
            gy = [general[:, pos[y], :].contiguous() for y in ys]
            px = torch.stack([fused_dense(gx[i], [self.ffm["ffm_x_%s_%s_%d" % (x, y, dim)] for y in ys], None)
                              for i, x in enumerate(xs)], dim=1).view(B, len(xs), len(ys), dim)       # [B, x, y, dim]
            py = torch.stack([fused_dense(gy[j], [self.ffm["ffm_y_%s_%s_%d" % (x, y, dim)] for x in xs], None)
                              .view(B, len(xs), dim) for j, y in enumerate(ys)], dim=2)               # [B, x, y, dim]
            ffm.append((px * py).reshape(B, -1))                                                      # x-major, as :14-21
        ffm = torch.cat(ffm, dim=-1) if len(ffm) > 1 else ffm[0]
        concated = torch.cat([reweight.reshape(B, n * 16), cross_term, mult, ffm] + din_embs, dim=-1)   # :122-123
        gate_input = G.index_select(1, bidx)[:, :, 16:].reshape(B, -1)                                # :126
        # PPNet-gated experts (:130-148)
        # layers that read the same tensor run as ONE GEMM over their kernels side by side (fused_dense): the first
        # expert layer of every expert and the first gate layer of every task all read `concated` (six Dense(relu));
        # the first PPNet gate layer of every (expert, level) reads `gate_input` (six Dense(relu))
        E, T, nu = C.num_experts, C.num_tasks, len(self.units)
        first = [self.experts["expert_output_%d_0" % i] for i in range(E)] + [self.task_gates["gate_%d_0" % i] for i in range(T)]
        first_out = torch.split(fused_dense(concated, first, "relu"), [l.units for l in first], dim=1)
        g1 = [self.experts["gate_%d_%d_1" % (i, j)] for i in range(E) for j in range(nu)]
        g1_out = torch.split(fused_dense(gate_input, g1, "relu"), [l.units for l in g1], dim=1)
        expert_outs = []
        for i in range(E):
            deep = concated
            for j in range(nu):
                g = self.experts["gate_%d_%d_2" % (i, j)](g1_out[i * nu + j]) * 2.0
                deep = g * (first_out[i] if j == 0 else self.experts["expert_output_%d_%d" % (i, j)](deep))
            expert_outs.append(deep)
        expert_concat = torch.stack(expert_outs, dim=1)                                               # [B, E, dim]
        mmoe = []
        for i in range(T):                                                                            # :153-164
            go = self.task_gates["gate_%d_1" % i](first_out[E + i])
            go = self.task_gates["gate_output_%d" % i](go).unsqueeze(-1)
            mmoe.append((expert_concat * go).sum(dim=1))
        # stay-time head: 400-way softmax + expectation over the bins (:167-179)
        ext = torch.cat([mmoe[0], self.cross(concated)], dim=-1)
        p = torch.softmax(self.staytime_output(ext), dim=-1)
        pred = p @ self.wt_bins
        pred = torch.where(pred < 0.0, torch.zeros_like(pred), pred)
        final_y = torch.cat([p, pred], dim=-1)                                                        # [B, 401]
        outs = {}
        for k, t in enumerate(C.task_names[1:], start=1):                                             # :181-191
            deep_logit = self.tower_deep["tower_deep_%s" % t](mmoe[k])
            outs[t] = self.tower_out[t](torch.cat([fm_logit, deep_logit], dim=1))
        train = {TASK_KEYS[0]: final_y, TASK_KEYS[1]: outs[C.task_names[1]], TASK_KEYS[2]: outs[C.task_names[2]]}
        predict = {TASK_KEYS[0]: pred, TASK_KEYS[1]: outs[C.task_names[1]], TASK_KEYS[2]: outs[C.task_names[2]]}
        return train, predict


def create_moe_sub_model(slots, seq_slots, deep_hidden_units):
    return VideoDnnSubModel(slots, seq_slots, deep_hidden_units)


# ------------------------------------------------------------------ losses (staytime/model.py:20-60)
_K_EPSILON = 1e-7          # tf.keras.backend.epsilon()


def custom_kl_loss(y_true, y_pred):
    yt = y_true[:, 0:C.multiclass_num].to(y_pred.dtype).clamp(_K_EPSILON, 1.0)
    yp = y_pred[:, 0:C.multiclass_num].clamp(_K_EPSILON, 1.0)
    return (yt * torch.log(yt / yp)).sum(dim=-1)


def cross_entropy(y_true, y_pred, a=1):
    y_true = y_true.to(torch.float32)
    return -y_true * torch.log(y_pred + 1e-6) - (a - y_true) * torch.log(1.0 - y_pred + 1e-6)


def mse_loss(y_true, y_pred):
    y = y_true.to(torch.float32)
    return ((torch.where(y > 2.0, torch.full_like(y, 2.0), y) - y_pred) ** 2).mean()


def huber_loss(y_true, y_pred, clip_delta=1.0):
    err = y_true - y_pred
    return torch.where(err.abs() < clip_delta, 0.5 * err * err, clip_delta * (err.abs() - 0.5 * clip_delta))


LOSSES = {TASK_KEYS[0]: custom_kl_loss, TASK_KEYS[1]: cross_entropy, TASK_KEYS[2]: cross_entropy}
LOSS_WEIGHTS = {TASK_KEYS[0]: 2.0, TASK_KEYS[1]: 2.0, TASK_KEYS[2]: 1.0}                     # model.py:85-87


class MtlNet(ComposedNet):
    """mtl_net(...) (staytime/VideoDnn.py:266-302): 32-d embeddings for every slot (combiner mean) plus the
    `[B, seq_max_len, 32]` sequence lookups of `seq_slots` (combiner None), sparse AdaGrad(0.005, g2sum 0.1,
    scale 0.1) (:233), feeding VideoDnnSubModel.  `train` / `predict` are the two graph outputs of the
    reference; `train_step` adds the compile() of staytime/model.py:72-90 (dense Adam 5e-4, weighted losses)."""
    dense_lr = 0.0005

    def __init__(self, slots, seq_slots, seq_max_len, dnn_hidden_units=(64, 32), bucket_size=81920, device="cuda:0",
                 seed=0, embedding_cls=None, group=None):
        self.slots, self.seq_slots = list(slots), list(seq_slots)
        cats = {s: category_column(s, bucket_size) for s in self.slots}                                  # :219-220
        # single-valued columns in sorted-slot order: the stacked gather output [B, n, 32] then IS the sub-model's
        # slot axis (mtl_net visits the slots sorted, :282,296) and no per-slot tensor is ever materialised
        cols = [embedding_column(cats[s], 32, combiner="mean", name="emb_col_%s" % s) for s in sorted(self.slots)]
        cols += [embedding_column(cats[s], 32, combiner=None, seq_max_len=seq_max_len, name="emb_col_seq_%s" % s)
                 for s in self.seq_slots]                                                                # :228-231
        super().__init__(cols, AdaGrad(learning_rate=0.005, initial_g2sum=0.1, initial_scale=0.1), "sparse_emb_input",
                         device, seed, embedding_cls, group)
        self.sub_model = VideoDnnSubModel(self.slots, self.seq_slots, dnn_hidden_units).to(device)

    def _embed(self, inputs):
        e = self.emb(inputs)
        st = getattr(self.emb, "last_stacked", None)
        want = ["emb_col_%s" % s for s in sorted(self.slots)]
        if st is not None and st[0] == want:
            embs = st[1]                                       # [B, n, 32], sorted-slot order, as gathered
        else:
            embs = {s: e["emb_col_%s" % s] for s in self.slots}
        seqs = {s: e["emb_col_seq_%s" % s] for s in self.seq_slots}
        return embs, seqs

    def train(self, inputs):
        embs, seqs = self._embed(inputs)
        return self.sub_model(embs, seqs)[0]

    def predict(self, inputs):
        with torch.no_grad():
            embs, seqs = self._embed(inputs)
            return self.sub_model(embs, seqs)[1]

    def _leaves(self, inputs):
        embs, seqs = self._embed(inputs)
        stacked = not isinstance(embs, dict)
        le = embs.detach().requires_grad_(True) if stacked else {s: v.detach().requires_grad_(True) for s, v in embs.items()}
        return le, {s: (v[0].detach().requires_grad_(True), v[1]) for s, v in seqs.items()}

    def _column_grads(self, x):
        le, ls = x
        if torch.is_tensor(le):                                # stacked [B, n, 32] leaf
            grads = {"emb_col_%s" % s: le.grad[:, i, :] for i, s in enumerate(sorted(self.slots))}
        else:
            grads = {"emb_col_%s" % s: v.grad for s, v in le.items()}
        grads.update({"emb_col_seq_%s" % s: v[0].grad for s, v in ls.items()})
        return grads

    def _forward(self, x, inputs):
        return self.sub_model(*x)[0]

    def _loss(self, out, labels):
        return sum(LOSS_WEIGHTS[k] * LOSSES[k](labels[k], out[k]).mean() for k in TASK_KEYS)


def mtl_net(slots, seq_slots, seq_max_len, dnn_hidden_units=(64, 32), **kw):
    net = MtlNet(slots, seq_slots, seq_max_len, dnn_hidden_units, **kw)
    return {"train": net.train, "predict": net.predict, "net": net}


def create_model_func(**kw):
    """staytime/model.py:68-92."""
    return mtl_net(C.SLOTS, C.SEQ_SLOTS, 50, dnn_hidden_units=(256, 128), **kw)
