"""Base of the composed nets (api.video_dnn.MtlNet, api.rough_rank_model.DssmNet, api.rank_ctr.RankCtrNet and the
AUTOINT model of api.builders): sparse embedding -> dense sub-model, trained by one `train_step`.

A composed net is any object with
    emb                         api.embedding.EmbeddingFeatures or api.sharded_embedding.ShardedEmbeddingFeatures
    sub_model                   the dense nn.Module
    opt, dense_optimizer()      its api.optim.DenseAdam: None until dense_optimizer() creates it (the lazily-built
                                layers must exist by then)
    predict(inputs)             a forward without gradients
    train_step(inputs, labels)  -> (loss, outputs)
api.graph.GraphedTrainStep and recommendsystem_b200.checkpoint work on any object with these.  ComposedNet supplies
them; a subclass states how the embedding outputs become the sub-model's inputs (and their gradients column
gradients again), the forward call and the loss.
"""
from __future__ import annotations

from typing import Dict

import torch

from .embedding import EmbeddingFeatures
from .optim import DenseAdam


class ComposedNet:
    dense_lr: float                    # learning rate of the dense Adam (betas 0.9 / 0.999, eps 1e-8)

    def __init__(self, cols, sparse_opt, name, device, seed, embedding_cls=None, group=None, id_map="mod"):
        # embedding_cls = api.sharded_embedding.ShardedEmbeddingFeatures (+ its process group): row-sharded tables
        # over the ranks, dense gradients averaged over them (staytime/parse.py:77-79); its group None is the default
        # process group
        E, kw = (embedding_cls, {"group": group}) if embedding_cls is not None else (EmbeddingFeatures, {})
        if id_map != "mod":
            kw["id_map"] = id_map
        self.emb = E(cols, sparse_opt, name, device=device, seed=seed, **kw)
        if embedding_cls is not None and group is None:
            import torch.distributed as dist
            group = dist.group.WORLD
        self.group = group
        self.opt = None

    def dense_optimizer(self) -> DenseAdam:
        """The dense Adam of sub_model, created at the first call: the lazily-built layers must exist."""
        if self.opt is None:
            self.opt = DenseAdam(self.sub_model.parameters(), lr=self.dense_lr, beta1=0.9, beta2=0.999, eps=1e-8,
                                 group=self.group)
        return self.opt

    def train_step(self, inputs, labels):
        """Embedding gather, forward, loss, dense Adam on sub_model, then the sparse push of the embedding gradients."""
        x = self._leaves(inputs)
        out = self._forward(x, inputs)
        opt = self.dense_optimizer()
        loss = self._loss(out, labels)
        opt.zero_grad()
        loss.backward()
        opt.step()
        self.emb.backward(self._column_grads(x))
        return loss.detach(), out.detach() if torch.is_tensor(out) else {k: v.detach() for k, v in out.items()}

    # ---- what differs between the nets
    def _leaves(self, inputs):
        """The sub-model's inputs: the embedding outputs detached into autograd leaves (dict column key -> leaf)."""
        return {k: v.detach().requires_grad_(True) for k, v in self.emb(inputs).items()}

    def _column_grads(self, x) -> Dict[str, torch.Tensor]:
        """d(loss)/d(embedding output) by column key, from the gradients of the leaves `x`."""
        return {k: v.grad for k, v in x.items()}

    def _forward(self, x, inputs):
        return self.sub_model(x)

    def _loss(self, out, labels) -> torch.Tensor:
        raise NotImplementedError
