"""FFM kernels at the edges of the shapes they are built for.

rs_ffm_fwd (ffm.cu) and the stash-free step (ffm_train.cu) keep one sample's F x F x D tile in shared memory, in a ring
of `nst` stages.  The largest tiles leave room for one stage only, so every wait on the ring's mbarriers flips its
phase; rows of more than 32 fields take the BIGF path (two id registers per lane, cold_mask bits up to 63); and the
gradient gather of the stash-free step is built for rows of 1, 2, 4 and 8 float4 per lane (NA).  These tests run
each of those cases against float64 restatements and the CPU oracle.
"""
import os
import re

import numpy as np
import pytest
import torch

from oracle import nfield as onf

SMEM = 232448          # 227 KB of shared memory per SM on B200
EPS32 = 2.0 ** -24
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "deeplearningrecommendationsystem_b200", "csrc")


def tile_bytes(F, D):
    """shared-memory bytes of one sample's tile: F rows of F*D floats, padded as ffm.cu / ffm_train.cu pad them"""
    dv = D // 4
    row_bytes = F * dv * 16
    pad = (dv * 16 - row_bytes) % 128 if dv < 8 else 0
    return F * (row_bytes + pad)


def fwd_stages(F, D):
    """ring stages of rs_ffm_fwd (ffm_fwd_launch, two CTAs per SM by default); 0 = the tile does not fit"""
    stage = tile_bytes(F, D)
    nst = (SMEM // 2 - 2048 - 1024) // stage
    if nst < 2:
        nst = (SMEM - 2048 - 1024) // stage
    return min(nst, 8)


def train_stages(F, D):
    """ring stages of ffm_single_kernel (rs_ffm_bwd_update)"""
    return min((SMEM - 6144) // tile_bytes(F, D), 8)


def test_stage_restatement_tracks_the_sources():
    """fwd_stages / train_stages restate the budgets of ffm.cu and ffm_train.cu; if those change, the shapes below that
    are meant to run a one-stage ring have to be re-derived."""
    def norm(name):
        with open(os.path.join(CSRC, name)) as f:
            return re.sub(r"\s+", " ", f.read())
    fwd, train = norm("ffm.cu"), norm("ffm_train.cu")
    assert "const size_t budget = 232448 / want_ctas - 2048 - 1024;" in fwd
    assert "int nst = (int)(budget / stage_bytes);" in fwd
    assert "if (nst < 2 && want_ctas == 2) nst = (int)((232448 - 2048 - 1024) / stage_bytes);" in fwd
    assert "int nst = (int)((232448 - 6144) / stage_bytes);" in train
    assert tile_bytes(14, 256) == 200704
    assert fwd_stages(14, 256) == 1 and fwd_stages(15, 256) == 0
    for F, D in ((48, 16), (64, 8)):
        assert fwd_stages(F, D) == 1 and train_stages(F, D) == 1, (F, D)


# ---------------------------------------------------------------------------------------------- forward with stash
@pytest.mark.gpu
@pytest.mark.parametrize("F,D", [(64, 4), (33, 8), (2, 256), (14, 256)])
def test_ffm_fwd_stash_at_shape_limits(F, D):
    """F = 64 (the most fields; BIGF), F = 33 (the first BIGF shape), D = 256, and F = 14 at D = 256: the largest tile
    that fits (200,704 B, one CTA per SM, one ring stage).  600 samples per launch: each CTA runs several of them
    through its ring.  cross against float64; the stash is an exact transposed copy with a zero diagonal."""
    from deeplearningrecommendationsystem_b200 import ops
    B = 600
    g = torch.Generator().manual_seed(F * 1000 + D)
    rows = [5 + 3 * f for f in range(F)]
    tabs = [torch.randn(r, F * D, generator=g) * 0.3 for r in rows]
    ids = torch.stack([torch.randint(0, r, (B,), generator=g) for r in rows], dim=1)
    ids[0], ids[1] = 0, torch.tensor(rows) - 1
    T = torch.stack([tabs[f][ids[:, f]] for f in range(F)], dim=1).view(B, F, F, D)
    Tt = T.transpose(1, 2)
    prod = (T.double() * Tt.double()).sum(3).triu(1)
    want = prod.sum((1, 2))
    S = (T.double() * Tt.double()).abs().sum(3).triu(1).sum((1, 2))
    keep = [t.cuda() for t in tabs]
    cross, stash = ops.ffm_fwd(ops.make_tables(keep), ids.cuda(), D, want_stash=True)
    ops.check_status()
    err = (cross.cpu().double() - want).abs()
    bound = 1e-5 * want.abs() + 4 * EPS32 * S
    assert bool((err <= bound).all()), f"max err / bound {float((err / bound).max()):.3f}"
    jac = Tt * (1.0 - torch.eye(F))[None, :, :, None]
    assert torch.equal(stash.cpu().view(B, F, F, D), jac)


@pytest.mark.gpu
def test_ffm_fwd_rejects_a_tile_that_does_not_fit():
    """F = 15, D = 256: a 230,400-byte tile is more than one CTA can hold"""
    from deeplearningrecommendationsystem_b200 import ops
    F, D = 15, 256
    keep = [torch.zeros(2, F * D, device="cuda") for _ in range(F)]
    with pytest.raises(RuntimeError, match="does not fit"):
        ops.ffm_fwd(ops.make_tables(keep), torch.zeros(4, F, dtype=torch.int64, device="cuda"), D, want_stash=True)


# ---------------------------------------------------------------------------------------------- stash-free SGD steps
@pytest.mark.gpu
@pytest.mark.parametrize("cards,D", [
    ([70000, 3, 50, 7, 1000, 24, 12, 301, 5], 16),                    # F*D = 144: NA = 2
    ([70000 if k == 40 else 5 + 13 * k for k in range(48)], 16),      # F = 48, F*D = 768: NA = 8, BIGF, one-stage ring
    ([70000 if k == 63 else 5 + 11 * k for k in range(64)], 8),       # F = 64: cold field 63 (cold_mask bit 63), one-stage ring
], ids=["F9xD16", "F48xD16", "F64xD8"])
def test_ffm_stash_free_steps_at_shape_limits(cards, D, monkeypatch):
    """Three SGD steps of FieldFFM with RS_FFM_RECOMPUTE=1 (stash-free: ffm_fwd_train + rs_ffm_bwd_update) and =0
    (rs_ffm_fwd with stash + rs_segment_update): bit-identical to each other, and equal to oracle.nfield.train_step.
    A field of >= 65536 rows makes the cold path run: its once-looked-up rows are updated in place by ffm_single_kernel,
    its slices of the other rows come from the cold-slice stash."""
    from deeplearningrecommendationsystem_b200 import ops
    from deeplearningrecommendationsystem_b200.nfield import FieldFFM
    from deeplearningrecommendationsystem_b200.optim import FusedRowOptimizer
    from deeplearningrecommendationsystem_b200.trainer import Trainer
    F, B, lr = len(cards), 1500, 0.3
    g = torch.Generator().manual_seed(F + D)
    ids = torch.stack([(torch.rand(B, generator=g) ** 2 * c).long().clamp_(max=c - 1) for c in cards], dim=1)
    ids[0], ids[1] = 0, torch.tensor(cards) - 1
    y = (torch.rand(B, 1, generator=g) < 0.3).float()
    out = {}
    for mode in ("1", "0"):
        monkeypatch.setenv("RS_FFM_RECOMPUTE", mode)
        m = FieldFFM(cards, D, fused=True, seed=9, device="cuda")
        tr = Trainer(m, torch.nn.BCELoss(), FusedRowOptimizer(m, torch.optim.SGD([m.bias], lr=lr), lr=lr, kind="sgd"))
        assert m._recompute == (mode == "1")
        assert m.cold_mask == sum(1 << f for f, c in enumerate(cards) if c >= 65536)
        table, bias = m.weight.detach().cpu().clone(), m.bias.detach().cpu().clone()
        offsets = torch.tensor(m.offsets_host)
        launches = ops.launches()
        preds = []
        for step in range(3):
            tr.train_loop(ids.cuda(), train_rating=y.cuda())
            preds.append(tr.predictions_train.detach().clone())
            if mode == "1":
                pred, loss = onf.train_step("ffm", table, bias, ids, offsets, y[:, 0], lr, fast=True)
                what = f"step {step + 1}"
                np.testing.assert_allclose(preds[-1].cpu().numpy()[:, 0], pred.numpy(), rtol=1e-5, atol=1e-6, err_msg=what)
                np.testing.assert_allclose(tr.train_loss.item(), loss.item(), rtol=1e-5, err_msg=what)
                np.testing.assert_allclose(m.weight.detach().cpu().numpy(), table.numpy(), rtol=1e-5, atol=2e-6, err_msg=what)
                np.testing.assert_allclose(m.bias.item(), bias.item(), rtol=1e-5, atol=1e-7, err_msg=what)
        ops.check_status()
        out[mode] = (m.weight.detach().clone(), preds, ops.launches() - launches)
        del m, tr
    assert all(torch.equal(a, b) for a, b in zip(out["1"][1], out["0"][1]))
    assert torch.equal(out["1"][0], out["0"][0])
    assert out["1"][2] != out["0"][2]           # the two runs really took different kernels
