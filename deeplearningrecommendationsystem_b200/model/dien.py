"""DIEN as the reference defines it (model/dien.py:8-81): a DIN-style attention with a smaller unit (3D->64->32->1)
that SCALES the history instead of pooling it, an nn.GRU(D, D) over the scaled sequence (h0 = 0), and
fc 2D->128->64->1->Sigmoid on [h_L, target].  This is a plain GRU on attention-scaled inputs, not the paper's AUGRU.

DIEN(..., evolution="augru") is the interest-evolution layer of the DIEN paper (Zhou et al., AAAI 2019) instead: the
attention weights a_t gate the GRU's update, u = a_t (1 - z), h_t = (1 - u) h_{t-1} + u n (torch's gate convention),
over the unscaled history, with the same nn.GRU weights.  It is an extension: the reference has no AUGRU, so its
parity is not pinned by the reference, only by the float64 restatement in tests/test_augru_gpu.py.  Both modes have the
same state_dict; the default (evolution="gru") is the reference's model.

DIEN(..., extractor=True, aux_weight=1.0) adds the paper's interest extractor and auxiliary loss (also extensions,
pinned by tests/test_dien_extractor_gpu.py):
  * interest_extractor, an nn.GRU(D, D) from h0 = 0 over the history embeddings e_0..e_{L-1}, gives states h_t; the
    attention rows are [h_0..h_{L-1} | e_target] and the evolution layer ("gru" or "augru") runs over the h_t;
  * L_aux = mean over b and t < L-1 of softplus(-<h_t, e_{t+1}>) + softplus(<h_t, e^_{t+1}>), with e^_{t+1} the
    embedding of an item drawn uniformly and redrawn while it equals hist[b, t+1] (L = 1 gives 0).  The draw is
    rs_dien_negatives' Philox stream keyed by a seed taken from torch's global generator at construction, with a
    device-resident epoch (a buffer kept out of state_dict) that every draw advances, so graph-replayed steps draw
    fresh negatives.  Histories are not masked: left-padded positions (id 0) enter the loss like any other.
  * The training objective is BCE + aux_weight * L_aux: in training (self.training and grad enabled, aux_weight > 0)
    the forward returns the predictions with aux_weight * L_aux attached, so that backpropagating the BCE of the
    predictions also backpropagates the auxiliary term with weight 1.  Trainer.train_loss stays the BCE alone;
    model.aux_loss holds the detached aux_weight * L_aux of the last training forward.  aux_weight = 0 is the paper's
    ablation: no negatives are drawn and no auxiliary kernel runs.  Eval and no_grad forwards draw nothing.
state_dict keys: din.item_embedding.weight, din.attention.{0,2,4}.*, interest_evolution.*_l0, fc.{0,2,4}.*
(+ interest_extractor.*_l0 with extractor=True)"""
import math

import torch
from torch import nn
from torch.nn.init import xavier_normal_

from . import _blocks as K
from .. import attention


class DIN(nn.Module, K.FusedRows):
    """Attention front half of DIEN: returns (history * attention weight (B, L, D), target embedding (B, D))."""

    def __init__(self, num_items, embed_size):
        super().__init__()
        self.item_embedding = nn.Embedding(num_items, embed_size)
        self.attention = nn.Sequential(nn.Linear(embed_size * 3, 64), nn.ReLU(), nn.Linear(64, 32), nn.ReLU(), nn.Linear(32, 1))
        xavier_normal_(self.item_embedding.weight.data)

    def _fused_groups(self):
        return [[self.item_embedding]]

    def forward(self, hist, target_item):
        rows = K.lookup(self.item_embedding.weight, torch.cat([hist, target_item.unsqueeze(1)], dim=1))
        return attention.din_attention(rows, self.attention, pool=False), rows[:, -1]

    def attend(self, hist, target_item):
        """-> (rows (B, L+1, D) = [history | target] embeddings, softmax attention weights (B, L))"""
        rows = K.lookup(self.item_embedding.weight, torch.cat([hist, target_item.unsqueeze(1)], dim=1))
        return rows, attention.din_attention_weights(rows, self.attention)


class _AttachAux(torch.autograd.Function):
    """pred unchanged; its backward also hands a gradient of 1 to the auxiliary term, so that BCE(pred).backward()
    backpropagates BCE + aux."""

    @staticmethod
    def forward(ctx, pred, aux):
        return pred.clone()

    @staticmethod
    def backward(ctx, g):
        return g, g.new_ones(())


class DIEN(nn.Module):
    """evolution: "gru" (the reference's GRU over the attention-scaled history) or "augru" (the paper's AUGRU).
    extractor: the paper's interest-extractor GRU and auxiliary loss; aux_weight (default 1.0 with the extractor, 0 =
    no auxiliary loss) weighs L_aux in the training objective.  See the module docstring."""

    def __init__(self, num_items, embed_size, evolution="gru", extractor=False, aux_weight=None):
        super().__init__()
        if evolution not in ("gru", "augru"):
            raise ValueError(f"DIEN: evolution must be 'gru' or 'augru', got {evolution!r}")
        if aux_weight is not None and not extractor:
            raise ValueError("DIEN: aux_weight needs extractor=True (the auxiliary loss supervises the extractor's states)")
        aux_weight = (1.0 if extractor else 0.0) if aux_weight is None else float(aux_weight)
        if not math.isfinite(aux_weight) or aux_weight < 0:
            raise ValueError(f"DIEN: aux_weight must be finite and >= 0, got {aux_weight!r}")
        if extractor and aux_weight > 0 and num_items < 2:
            raise ValueError(f"DIEN: the auxiliary loss needs num_items >= 2 (a negative distinct from the clicked item), "
                             f"got {num_items}")
        self.evolution, self.extractor, self.aux_weight = evolution, bool(extractor), aux_weight
        self.din = DIN(num_items, embed_size)
        self.interest_evolution = nn.GRU(embed_size, embed_size, batch_first=True)
        self.fc = nn.Sequential(nn.Linear(embed_size * 2, 128), nn.ReLU(), nn.Linear(128, 64), nn.ReLU(), nn.Linear(64, 1),
                                nn.Sigmoid())
        self.aux_loss = None
        if self.extractor:
            self.num_items = num_items
            self.interest_extractor = nn.GRU(embed_size, embed_size, batch_first=True)
            self.aux_seed = int(torch.randint(0, 2 ** 63 - 1, (1,), dtype=torch.int64))
            self.register_buffer("aux_epoch", torch.zeros((), dtype=torch.int64), persistent=False)

    def fuse_embedding_updates(self):
        """opt-in fused sparse rows for the item table (see model/_blocks.RowSink); FusedRowOptimizer finds self.din"""
        self.din.fuse_embedding_updates()
        return self

    def forward(self, hist, target_item):
        if self.extractor:
            return self._forward_extractor(hist, target_item)
        if self.evolution == "augru":
            rows, w = self.din.attend(hist, target_item)
            final_interest = attention.augru_last_hidden(rows[:, :-1], w, self.interest_evolution)        # (B, D)
            return self.fc(torch.cat([final_interest, rows[:, -1]], dim=-1))
        att_hist, target_embed = self.din(hist, target_item)
        final_interest = attention.gru_last_hidden(att_hist, self.interest_evolution)                  # (B, D)
        return self.fc(torch.cat([final_interest, target_embed], dim=-1))

    def _forward_extractor(self, hist, target_item):
        from .. import ops
        L = hist.shape[1]
        aux_on = self.training and torch.is_grad_enabled() and self.aux_weight > 0
        ids = [hist, target_item.unsqueeze(1)]
        if aux_on:
            ids.append(ops.dien_negatives(hist, self.num_items, self.aux_seed, self.aux_epoch))
            self.aux_epoch.add_(1)
        # one lookup (one gather, one sort in the backward): [history | target | negatives] (B, 2L, D) in training
        rows = K.lookup(self.din.item_embedding.weight, torch.cat(ids, dim=1))
        hs = attention.gru_sequence(rows[:, :L], self.interest_extractor)                              # (B, L, D)
        target_embed = rows[:, L]
        att_rows = torch.cat([hs, target_embed.unsqueeze(1)], dim=1)
        if self.evolution == "augru":
            w = attention.din_attention_weights(att_rows, self.din.attention)
            final_interest = attention.augru_last_hidden(hs, w, self.interest_evolution)
        else:
            att_hist = attention.din_attention(att_rows, self.din.attention, pool=False)
            final_interest = attention.gru_last_hidden(att_hist, self.interest_evolution)
        pred = self.fc(torch.cat([final_interest, target_embed], dim=-1))
        if not aux_on:
            return pred
        aux = attention.dien_aux_loss(hs, rows[:, 1:L], rows[:, L + 1:]) * self.aux_weight
        self.aux_loss = aux.detach()
        return _AttachAux.apply(pred, aux)

    def recommendation(self, num_users, num_items, hist_list, k):
        device = next(self.parameters()).device
        return K.rank_catalogue(K.history_scores(self, hist_list, num_items, device), num_users, num_items, k)
