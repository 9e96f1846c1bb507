"""DIEN as the reference defines it (model/dien.py:8-81): a DIN-style attention with a smaller unit (3D->64->32->1)
that SCALES the history instead of pooling it, an nn.GRU(D, D) over the scaled sequence (h0 = 0), and
fc 2D->128->64->1->Sigmoid on [h_L, target].  This is a plain GRU on attention-scaled inputs, not the paper's AUGRU.

DIEN(..., evolution="augru") is the interest-evolution layer of the DIEN paper (Zhou et al., AAAI 2019) instead: the
attention weights a_t gate the GRU's update, u = a_t (1 - z), h_t = (1 - u) h_{t-1} + u n (torch's gate convention),
over the unscaled history, with the same nn.GRU weights.  It is an extension: the reference has no AUGRU, so its
parity is not pinned by the reference, only by the float64 restatement in tests/test_augru_gpu.py.  Both modes have the
same state_dict; the default (evolution="gru") is the reference's model.
state_dict keys: din.item_embedding.weight, din.attention.{0,2,4}.*, interest_evolution.*_l0, fc.{0,2,4}.*"""
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


class DIEN(nn.Module):
    """evolution: "gru" (the reference's GRU over the attention-scaled history) or "augru" (the paper's AUGRU)."""

    def __init__(self, num_items, embed_size, evolution="gru"):
        super().__init__()
        if evolution not in ("gru", "augru"):
            raise ValueError(f"DIEN: evolution must be 'gru' or 'augru', got {evolution!r}")
        self.evolution = evolution
        self.din = DIN(num_items, embed_size)
        self.interest_evolution = nn.GRU(embed_size, embed_size, batch_first=True)
        self.fc = nn.Sequential(nn.Linear(embed_size * 2, 128), nn.ReLU(), nn.Linear(128, 64), nn.ReLU(), nn.Linear(64, 1),
                                nn.Sigmoid())

    def fuse_embedding_updates(self):
        """opt-in fused sparse rows for the item table (see model/_blocks.RowSink); FusedRowOptimizer finds self.din"""
        self.din.fuse_embedding_updates()
        return self

    def forward(self, hist, target_item):
        if self.evolution == "augru":
            rows, w = self.din.attend(hist, target_item)
            final_interest = attention.augru_last_hidden(rows[:, :-1], w, self.interest_evolution)        # (B, D)
            return self.fc(torch.cat([final_interest, rows[:, -1]], dim=-1))
        att_hist, target_embed = self.din(hist, target_item)
        final_interest = attention.gru_last_hidden(att_hist, self.interest_evolution)                  # (B, D)
        return self.fc(torch.cat([final_interest, target_embed], dim=-1))

    def recommendation(self, num_users, num_items, hist_list, k):
        device = next(self.parameters()).device
        return K.rank_catalogue(K.history_scores(self, hist_list, num_items, device), num_users, num_items, k)
