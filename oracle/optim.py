"""Optimiser arithmetic restated on CPU (fp32).  TEST INFRASTRUCTURE ONLY -- see oracle/__init__.py.

``adam_dense`` follows torch.optim.Adam's single-tensor path, which is what the reference scripts run
(`optim.Adam(model.parameters(), lr, weight_decay=1e-5)`, scripts/deepfm.py:55, stepped at
trainer/trainer.py:39): L2 decay folded into the gradient, EVERY row of every table moves every step.
``sgd_rows`` / ``adam_rows`` are the row-sparse updates the fused kernels implement; sgd_rows is exactly
equal to dense SGD (momentum 0, wd 0); adam_rows is an extension with no reference counterpart
("parity unpinned": its oracle is this file, not the reference).
"""
import math

import torch


def adam_dense(p, g, m, v, step, lr=1e-3, b1=0.9, b2=0.999, eps=1e-8, wd=0.0):
    """One torch.optim.Adam step (amsgrad off).  `step` is the 1-based step count.  Returns (p, m, v)."""
    if wd != 0.0:
        g = g + wd * p
    m = torch.lerp(m, g, 1.0 - b1)
    v = b2 * v + (1.0 - b2) * g * g
    bc1 = 1.0 - b1 ** step
    bc2 = 1.0 - b2 ** step
    denom = v.sqrt() / math.sqrt(bc2) + eps
    return p - (lr / bc1) * (m / denom), m, v


def segment_sum_rows(ids, G):
    """Sum the rows of G (N, W) that share an id, visiting them in ascending position -- the order of the
    reference's CPU embedding_dense_backward (sequential index_add).  Returns (unique_ids, sums)."""
    uniq, inv = torch.unique(ids, sorted=True, return_inverse=True)
    out = torch.zeros(uniq.numel(), G.shape[1], dtype=G.dtype)
    out.index_add_(0, inv, G)
    return uniq, out


def sgd_rows(table, ids, G, lr):
    """table[u] -= lr * sum_{p: ids[p]==u} G[p]  (in place) -- equals dense SGD on the dense gradient."""
    uniq, gs = segment_sum_rows(ids, G)
    table[uniq] -= lr * gs
    return table


def adam_rows(table, m, v, ids, G, step, lr=1e-3, b1=0.9, b2=0.999, eps=1e-8, wd=0.0):
    """Lazy (row-sparse) Adam: only touched rows update their moments and weights.  wd: L2 decay folded into the
    summed gradient of each touched row, as torch.optim.Adam(weight_decay=wd) does."""
    uniq, g = segment_sum_rows(ids, G)
    if wd != 0.0:
        g = g.add(table[uniq], alpha=wd)
    mu = torch.lerp(m[uniq], g, 1.0 - b1)
    vu = b2 * v[uniq] + (1.0 - b2) * g * g
    bc1 = 1.0 - b1 ** step
    bc2 = 1.0 - b2 ** step
    table[uniq] -= (lr / bc1) * (mu / (vu.sqrt() / math.sqrt(bc2) + eps))
    m[uniq] = mu
    v[uniq] = vu
    return table, m, v
