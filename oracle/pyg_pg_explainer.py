"""ORACLE -- TEST INFRASTRUCTURE ONLY.  Never imported by the product package.

PyG's ``PGExplainer`` for graph-level, "phenomenon" explanations, on top of ``oracle/pyg_explain.py``
(``MaskedOracleLeakDetector``, used unchanged).  Restated from PyG 2.x's published source
``torch_geometric/explain/algorithm/pg_explainer.py``, unpinned like the rest of the restatement:

    coeffs = {'edge_size': 0.05, 'edge_ent': 1.0, 'temp': [5.0, 2.0], 'bias': 0.01}
    __init__(epochs, lr=0.003, **kwargs):  mlp = Sequential(Linear(-1, 64), ReLU(), Linear(64, 1))
                                           optimizer = Adam(mlp.parameters(), lr=lr); _curr_epoch = -1
    train(epoch, model, x, edge_index, *, target, index=None, **kwargs):
        z = get_embeddings(model, x, edge_index, **kwargs)[-1]
        optimizer.zero_grad(); temperature = _get_temperature(epoch)
        inputs = _get_inputs(z, edge_index, index); logits = mlp(inputs).view(-1)
        edge_mask = _concrete_sample(logits, temperature)
        set_masks(model, edge_mask, edge_index, apply_sigmoid=True)
        y_hat, y = model(x, edge_index, **kwargs), target
        loss = _loss(y_hat, y, edge_mask); loss.backward(); optimizer.step()
        clear_masks(model); _curr_epoch = epoch; return float(loss)
    forward(model, x, edge_index, *, target, index=None, **kwargs):
        if _curr_epoch < epochs - 1: raise ValueError("... is not yet fully trained ...")
        z = get_embeddings(...)[-1]; inputs = _get_inputs(z, edge_index, index); logits = mlp(inputs).view(-1)
        edge_mask = _post_process_mask(logits, hard_edge_mask=None, apply_sigmoid=True)
    _get_inputs(embedding, edge_index, index=None):  cat([embedding[edge_index[0]], embedding[edge_index[1]]], -1)
    _get_temperature(epoch):  temp[0] * pow(temp[1] / temp[0], epoch / epochs)
    _concrete_sample(logits, temperature=1.0, training=True):
        eps = (1 - 2 * bias) * torch.rand_like(logits) + bias
        return (eps.log() - (1 - eps).log() + logits) / temperature
    _loss(y_hat, y, edge_mask):  loss = cross_entropy(y_hat, y)       (multiclass, raw outputs)
        mask = edge_mask.sigmoid(); size_loss = mask.sum() * edge_size
        mask = 0.99 * mask + 0.005; mask_ent = -mask * mask.log() - (1 - mask) * (1 - mask).log()
        return loss + size_loss + mask_ent.mean() * edge_ent

``get_embeddings`` (``torch_geometric/utils/embedding.py``) registers a forward hook on every ``MessagePassing``
module, runs the model in eval mode under ``no_grad`` and returns the hooked outputs: ``[-1]`` is the last
``GCNConv``'s output, before the ReLU and dropout the detector applies after it.  It is taken here the same way, by a
forward hook on the oracle's last conv.  PyG's ``Linear(-1, 64)`` materialises with ``torch.nn.Linear``'s
initialisation.  ``torch.rand_like`` is replaced by the ``uniform`` argument, so a test can replay the device's draws.
A batch of B windows is PyG's run on their disjoint union (the oracle's replicated ``edge_index``): the mask is (B, E)
laid out window by window, the cross-entropy is the mean over the windows, and both regularisers run over all B E
edges.  PyG's ``float(loss)`` is returned as the 0-d tensor.
"""
from __future__ import annotations

from typing import Optional

import torch
import torch.nn.functional as F


class PGExplainerOracle(torch.nn.Module):
    coeffs = {"edge_size": 0.05, "edge_ent": 1.0, "temp": (5.0, 2.0), "bias": 0.01}

    def __init__(self, node_dim: int, epochs: int, lr: float = 0.003, **coeffs) -> None:
        super().__init__()
        self.epochs, self.lr = int(epochs), float(lr)
        self.coeffs = {**PGExplainerOracle.coeffs, **coeffs}
        self.mlp = torch.nn.Sequential(torch.nn.Linear(2 * node_dim, 64), torch.nn.ReLU(), torch.nn.Linear(64, 1))
        self.optimizer = torch.optim.Adam(self.mlp.parameters(), lr=self.lr)
        self._curr_epoch = -1

    # --- PyG's helpers
    def _get_temperature(self, epoch: int) -> float:
        t0, t1 = self.coeffs["temp"]
        return t0 * pow(t1 / t0, epoch / self.epochs)

    def _concrete_sample(self, logits: torch.Tensor, temperature: float, uniform: torch.Tensor) -> torch.Tensor:
        bias = self.coeffs["bias"]
        eps = (1 - 2 * bias) * uniform.to(logits.dtype).reshape(logits.shape) + bias
        return (eps.log() - (1 - eps).log() + logits) / temperature

    @staticmethod
    def _get_inputs(embedding: torch.Tensor, edge_index: torch.Tensor) -> torch.Tensor:
        return torch.cat([embedding[edge_index[0]], embedding[edge_index[1]]], dim=-1)

    def _loss(self, y_hat: torch.Tensor, y: torch.Tensor, edge_mask: torch.Tensor) -> torch.Tensor:
        loss = F.cross_entropy(y_hat, y)
        mask = edge_mask.sigmoid()
        size_loss = mask.sum() * self.coeffs["edge_size"]
        mask = 0.99 * mask + 0.005
        mask_ent = -mask * mask.log() - (1 - mask) * (1 - mask).log()
        return loss + size_loss + mask_ent.mean() * self.coeffs["edge_ent"]

    # --- the model side: get_embeddings and the disjoint union of the B windows
    @staticmethod
    def get_embeddings(model, h_s: torch.Tensor) -> torch.Tensor:
        out = []
        handle = model.convs[-1].register_forward_hook(lambda mod, inp, o: out.append(o))
        training = model.training
        model.eval()
        try:
            with torch.no_grad():
                model.gnn_stack(h_s)
        finally:
            model.train(training)
            handle.remove()
        return out[-1]

    @staticmethod
    def batched_edge_index(model, b: int) -> torch.Tensor:
        e = model.edge_index_single.size(1)
        off = torch.arange(b).repeat_interleave(e) * model.num_nodes
        return model.edge_index_single.repeat(1, b) + off.unsqueeze(0)

    def logits(self, model, h_s: torch.Tensor) -> torch.Tensor:
        """The edge network's logits (B, E) on ``h_s``'s windows."""
        z = self.get_embeddings(model, h_s)
        return self.mlp(self._get_inputs(z, self.batched_edge_index(model, h_s.shape[0]))).view(h_s.shape[0], -1)

    def train(self, epoch, model=None, h_s: Optional[torch.Tensor] = None, target: Optional[torch.Tensor] = None,
              uniform: Optional[torch.Tensor] = None):
        if isinstance(epoch, bool) and model is None:
            return super().train(epoch)
        self.optimizer.zero_grad()
        temperature = self._get_temperature(epoch)
        logits = self.logits(model, h_s)
        edge_mask = self._concrete_sample(logits, temperature, uniform)
        y_hat = model.gnn_stack(h_s, edge_mask=edge_mask.sigmoid())       # set_masks(..., apply_sigmoid=True)
        loss = self._loss(y_hat, target, edge_mask.reshape(-1))
        loss.backward()
        self.optimizer.step()
        self._curr_epoch = epoch
        return loss.detach()

    def forward(self, model, h_s: torch.Tensor) -> torch.Tensor:
        if self._curr_epoch < self.epochs - 1:
            raise ValueError(f"'{type(self).__name__}' is not yet fully trained (got {self._curr_epoch + 1} epochs from "
                             f"{self.epochs} epochs)")
        with torch.no_grad():
            return self.logits(model, h_s).sigmoid()
