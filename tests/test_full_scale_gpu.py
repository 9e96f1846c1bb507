"""The C2 (FM + FFM on the Criteo cardinalities) and C5 (MF on two 100 M-row tables) train steps at their real table
sizes, each step checked against a sparse float64 reference of the same SGD step.

Every other test caps the cardinalities, so no kernel there ever addresses a row past 2^31 floats.  Here the FFM table
is 33.8 M rows x 416 floats (1.4e10 floats, 56 GB) and the MF table 2e8 rows x 64 floats (1.3e10 floats, 51 GB): a row
offset truncated to 32 bits would land inside the same allocation, fault nothing, and update the wrong row.  Each step
is checked three ways: predictions, loss and bias; every element of every row the batch touches; and bit-identity of
the rows it must not touch -- a seeded sample of over a million rows and the rows a 32-bit wrap of a touched row's
offset would hit instead.

The reference (sparse_sgd_reference) touches only the rows the batch looks up, so it runs at these sizes; the CPU test
at the top of this file pins it against the dense oracles (oracle.nfield.train_step, oracle.ml100k.mf).
"""
import gc
import sys
import time
import traceback

import numpy as np
import pytest
import torch

from oracle import interactions as OI, ml100k, nfield as onf

C2_CARDS = [1460, 583, 10131227, 2202608, 305, 24, 12517, 633, 3, 93145, 5683, 8351593, 3194, 27, 14992, 5461306, 10, 5652,
            2173, 4, 7046547, 18, 15, 286181, 105, 142572]
C5_ROWS = 100_000_000
D, B, LR = 16, 65536, 0.05
EPS32 = 2.0 ** -24
GUARD_SAMPLE = 1_000_000          # untouched rows compared bit for bit after every step (at least)


# ---------------------------------------------------------------------------------------------- sparse float64 reference
def sparse_sgd_reference(kind, rows, inv, y, lr, bias=None, dim=None, chunk=4096):
    """One SGD step of FM / FFM / MF with BCE-mean loss, in float64, over the rows a batch touches.

    rows (U, W): the distinct table rows the batch looks up, as they were before the step.  inv (B, F): index into
    `rows` of lookup (b, i).  y: B labels.  bias: the scalar bias before the step (FM / FFM), None for MF (no bias).
    dim: D of the FFM row (F slots of D floats).  Logits follow oracle.nfield.fm_logit / ffm_logit and oracle.ml100k.mf.
    Returns a dict: pred (B,), loss, rows (U, W) after the step, grad (U, W) = summed gradient, absg (U, W) = the L1 mass
    the element's fp32 gradient is formed from: the sum over its terms of |d loss / d logit| times the L1 mass of the
    Jacobian element (FM: sum_f e_f - e_i is formed from an fp32 sum over the fields that can cancel, so its mass is
    sum_f |e_f|, not its value; FFM and MF: a single table value), bias after the step (None for MF).  Stock torch ops
    only; runs where `rows` is.
    """
    nb, F = inv.shape
    U, W = rows.shape
    dev = rows.device
    y64 = y.reshape(-1).to(dev, torch.float64)
    grad = torch.zeros(U, W, dtype=torch.float64, device=dev)
    absg = torch.zeros(U, W, dtype=torch.float64, device=dev)
    pred = torch.empty(nb, dtype=torch.float64, device=dev)
    loss = torch.zeros((), dtype=torch.float64, device=dev)
    gsum = torch.zeros((), dtype=torch.float64, device=dev)
    b0 = 0.0 if bias is None else float(bias)
    if kind == "ffm":
        off_diag = (1.0 - torch.eye(F, dtype=torch.float64, device=dev))[None, :, :, None]
    for s in range(0, nb, chunk):
        idx = inv[s:s + chunk]
        c = idx.shape[0]
        E = rows[idx].double()                                     # (c, F, W)
        mass = None
        if kind == "fm":
            tot = E.sum(1)
            logit = 0.5 * (tot * tot - (E * E).sum(1)).sum(1)
            jac = tot.unsqueeze(1) - E                             # d logit / d e_i = sum_f e_f - e_i
            mass = E.abs().sum(1, keepdim=True).expand_as(E)      # the fp32 sum of the F rows can cancel
        elif kind == "mf":
            logit = (E[:, 0] * E[:, 1]).sum(1)
            jac = E.flip(1)                                        # d <u, v> / du = v, d / dv = u
        elif kind == "ffm":
            T = E.view(c, F, F, dim)                               # T[b, i, j] = v_{i,j}: row of field i, slot j
            Tt = T.transpose(1, 2)                                 # Tt[b, i, j] = v_{j,i}
            logit = (T * Tt).sum(3).triu(1).sum((1, 2))            # sum_{i<j} <v_{i,j}, v_{j,i}>
            jac = (Tt * off_diag).reshape(c, F, W)                 # slot j of row (b, i) gets v_{j,i}; its own slot 0
        else:
            raise ValueError(kind)
        p = torch.sigmoid(logit + b0)
        yc = y64[s:s + c]
        loss += -(yc * torch.clamp(torch.log(p), min=-100.0) + (1.0 - yc) * torch.clamp(torch.log(1.0 - p), min=-100.0)).sum()
        g = (p - yc) / nb                                          # d mean-BCE / d logit
        terms = (g[:, None, None] * jac).reshape(-1, W)
        flat = idx.reshape(-1)
        grad.index_add_(0, flat, terms)
        absg.index_add_(0, flat, terms.abs() if kind != "fm" else (g.abs()[:, None, None] * mass).reshape(-1, W))
        gsum += g.sum()
        pred[s:s + c] = p
        del E, jac, terms, mass
    return {"pred": pred, "loss": loss / nb, "rows": rows.double() - lr * grad, "grad": grad, "absg": absg,
            "bias": None if bias is None else b0 - lr * float(gsum)}


def _xavier_like(cards, width, row_dim, g):
    return torch.cat([torch.randn(c, width, generator=g) * (2.0 / (c + row_dim)) ** 0.5 for c in cards])


@pytest.mark.parametrize("kind", ["fm", "ffm", "mf"])
def test_sparse_reference_matches_dense_oracle(kind):
    """The reference above against the dense-gradient oracles on capped cardinalities, both in float64: predictions,
    loss, bias, every touched row -- and the rows the batch does not touch are left alone by the oracle's dense SGD."""
    torch.manual_seed(0)
    g = torch.Generator().manual_seed(17)
    nb, lr = 700, 0.5
    if kind == "mf":
        cards, dim, width = [300, 500], 64, 64
    else:
        cards, dim = [3, 50, 7, 1000, 24, 12, 301, 5], (16 if kind == "fm" else 4)
        width = dim if kind == "fm" else len(cards) * dim
    table = _xavier_like(cards, width, dim, g).double()
    offsets = torch.tensor([sum(cards[:k]) for k in range(len(cards))])
    ids = torch.stack([(torch.rand(nb, generator=g) ** 3 * c).long().clamp_(max=c - 1) for c in cards], dim=1)
    ids[0], ids[1] = 0, torch.tensor(cards) - 1
    y = (torch.rand(nb, generator=g) < 0.3).double()
    keys = ids + offsets
    uniq, inv = torch.unique(keys, return_inverse=True)
    bias0 = torch.tensor([0.07], dtype=torch.float64)
    ref = sparse_sgd_reference(kind, table[uniq], inv, y, lr, None if kind == "mf" else float(bias0), dim=dim)
    dense = table.clone()
    if kind == "mf":
        sd = {"user_embeddings.weight": dense[:cards[0]].clone().requires_grad_(True),
              "item_embeddings.weight": dense[cards[0]:].clone().requires_grad_(True)}
        pred = ml100k.mf(sd, ids[:, 0], ids[:, 1])
        loss = OI.bce(pred, y)
        gu, gi = torch.autograd.grad(loss, list(sd.values()))
        dense -= lr * torch.cat([gu, gi])
        want_bias = None
    else:
        bias = bias0.clone()
        pred, loss = onf.train_step(kind, dense, bias, ids, offsets, y, lr)
        want_bias = float(bias)
    np.testing.assert_allclose(ref["pred"].numpy(), pred.detach().numpy(), rtol=1e-12, atol=1e-15)
    np.testing.assert_allclose(float(ref["loss"]), float(loss.detach()), rtol=1e-12)
    if want_bias is not None:
        np.testing.assert_allclose(ref["bias"], want_bias, rtol=1e-12)
    np.testing.assert_allclose(ref["rows"].numpy(), dense[uniq].numpy(), rtol=1e-12, atol=1e-15)
    untouched = torch.ones(table.shape[0], dtype=torch.bool)
    untouched[uniq] = False
    assert torch.equal(dense[untouched], table[untouched])
    # the |term| sums bound the summed gradient
    assert bool((ref["absg"] >= ref["grad"].abs()).all())


# ---------------------------------------------------------------------------------------------- batches and guard rows
def zipf_ids(c, shape, g, device, a=1.05):
    """inverse CDF of a continuous power law with exponent a, truncated to [1, c] (bench.py's zipf ids)"""
    u = torch.rand(shape, generator=g, device=device, dtype=torch.float64)
    x = ((c ** (1 - a) - 1) * u + 1) ** (1 / (1 - a))
    return (x.floor().long() - 1).clamp_(0, c - 1)


def make_batch(cards, dist, seed, nb=B):
    """(nb, F) local ids drawn as bench.py draws them, with samples pinned to row 0 and to row card - 1 of every field
    (the last row of the last field is the highest address in the table), and Bernoulli(0.3) labels."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    cols = [zipf_ids(c, (nb,), g, "cuda") if dist == "zipf" else torch.randint(0, c, (nb,), generator=g, device="cuda") for c in cards]
    ids = torch.stack(cols, dim=1).contiguous()
    last = torch.tensor(cards, device="cuda") - 1
    ids[0], ids[nb // 2] = 0, 0
    ids[1], ids[nb - 1], ids[nb // 3] = last, last, last
    y = (torch.rand(nb, generator=g, device="cuda") < 0.3).float()
    return ids, y


def guard_sample(cards, seed, device):
    """sorted distinct rows of the concatenated table: a seeded sample of about 1.1 GUARD_SAMPLE rows spread over every
    field in proportion to its size, at least 1000 (or all) rows of each"""
    total = sum(cards)
    g = torch.Generator(device=device).manual_seed(seed)
    want = int(GUARD_SAMPLE * 1.1)
    parts, o = [], 0
    for c in cards:
        k = max(1000, want * c // total)
        parts.append(o + (torch.arange(c, device=device) if k >= c else torch.randint(0, c, (k,), generator=g, device=device)))
        o += c
    return torch.unique(torch.cat(parts))


def wrap_images(rows, base, width):
    """the rows that hold float offset (o mod 2^32) and (o mod 2^31) and byte offset (4 o mod 2^32) from `base`, where
    o = (rows - base) * width is the float offset of each row from that base: where a 32-bit offset would land"""
    o = (rows - base) * width
    return torch.cat([base + wrapped // width for wrapped in (o % (1 << 32), o % (1 << 31), (4 * o) % (1 << 32) // 4)])


def guard_rows(cards, width, uniq, seed):
    """Sorted distinct global rows the step must leave bit-identical: a seeded sample of >= GUARD_SAMPLE rows spread over
    every field, plus the wrap images of every touched row relative to the concatenated table and to the row's own
    field, minus the touched rows themselves."""
    dev = uniq.device
    total = sum(cards)
    offs = torch.tensor([sum(cards[:k]) for k in range(len(cards))], device=dev)
    sample = guard_sample(cards, seed, dev)
    sample = sample[~torch.isin(sample, uniq)]
    assert sample.numel() >= GUARD_SAMPLE, sample.numel()
    base = offs[torch.searchsorted(offs, uniq, right=True) - 1]
    images = torch.unique(torch.cat([wrap_images(uniq, b0, width) for b0 in (torch.zeros_like(uniq), base)]))
    images = images[~torch.isin(images, uniq)]
    assert images.numel() == 0 or int(images.max()) < total
    return torch.unique(torch.cat([sample, images])), int(images.numel())


# ---------------------------------------------------------------------------------------------- per-step checks
def assert_rows_match(got, ref, lr, what, chunk=1 << 17):
    """|w_gpu - w64| <= 1e-6 |w64| + lr (1e-5 |g64| + 4 eps32 S) for every element (S = ref["absg"], the L1 mass the
    gradient is formed from): the scaled floor of test_segment_grad_and_sgd -- a fp32 sum of n terms carries a few ulp of
    their L1 mass."""
    worst = 0.0
    for s in range(0, got.shape[0], chunk):
        w64, g64, S = ref["rows"][s:s + chunk], ref["grad"][s:s + chunk], ref["absg"][s:s + chunk]
        err = (got[s:s + chunk].double() - w64).abs()
        bound = 1e-6 * w64.abs() + lr * (1e-5 * g64.abs() + 4 * EPS32 * S)
        ratio = err / bound.clamp_min(1e-300)
        bad = err > bound
        if bool(bad.any()):
            r, e = (int(v) for v in bad.nonzero()[0])
            raise AssertionError(f"{what}: {int(bad.sum())} table elements outside the bound; first at touched row {s + r}, "
                                 f"element {e}: gpu {float(got[s + r, e])!r} want {float(w64[r, e])!r} "
                                 f"bound {float(bound[r, e]):.3e} (|g| {float(g64[r, e].abs()):.3e}, S {float(S[r, e]):.3e})")
        worst = max(worst, float(ratio.max()))
    return worst


def run_steps(kind, model, tr, inputs, y, keys, width, dim, steps=2):
    """`steps` SGD steps of Trainer.train_loop on the same batch.  Before each step the touched rows are read back; after
    it the step is compared with sparse_sgd_reference started from those rows (so every step is checked on its own)."""
    from deeplearningrecommendationsystem_b200 import ops
    uniq, inv = torch.unique(keys, return_inverse=True)
    guard, n_images = guard_rows(model.cards, width, uniq, seed=5)
    snap = model.weight.data[guard].view(torch.int32).clone()
    has_bias = kind != "mf"
    worst = []
    for step in range(1, steps + 1):
        before = model.weight.data[uniq].clone()
        bias0 = float(model.bias.detach()) if has_bias else None
        tr.train_loop(*inputs, train_rating=y)
        ops.check_status()
        ref = sparse_sgd_reference(kind, before, inv, y, LR, bias0, dim=dim)
        del before
        what = f"{kind} step {step}"
        np.testing.assert_allclose(tr.predictions_train.detach().reshape(-1).cpu().numpy(), ref["pred"].cpu().numpy(),
                                   rtol=1e-5, atol=1e-6, err_msg=what)
        np.testing.assert_allclose(float(tr.train_loss), float(ref["loss"]), rtol=1e-5, err_msg=what)
        if has_bias:
            np.testing.assert_allclose(float(model.bias.detach()), ref["bias"], rtol=1e-5, err_msg=what)
        worst.append(assert_rows_match(model.weight.data[uniq], ref, LR, what))
        del ref
        same = model.weight.data[guard].view(torch.int32) == snap
        if not bool(same.all()):
            r = int((~same.all(1)).nonzero()[0])
            raise AssertionError(f"{what}: {int((~same.all(1)).sum())} of {guard.numel()} untouched rows changed, first global row "
                                 f"{int(guard[r])} ({n_images} of the guard rows are 32-bit wrap images of touched rows)")
    return {"touched_rows": int(uniq.numel()), "guard_rows": int(guard.numel()), "wrap_images": n_images,
            "worst_err_over_bound": max(worst)}


# ---------------------------------------------------------------------------------------------- GPU cases
@pytest.fixture
def big_case():
    """Frees the case's model before the next test -- also when the test failed: pytest keeps the traceback of the
    last failure (sys.last_traceback), whose frames would otherwise pin tens of GB of device memory."""
    held = {}
    t0 = time.perf_counter()
    torch.cuda.reset_peak_memory_stats()
    yield held
    tb = getattr(sys, "last_traceback", None)
    if tb is not None:
        traceback.clear_frames(tb)
    info = held.pop("info", None)
    held.clear()
    gc.collect()
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() / 1e9
    torch.cuda.empty_cache()
    print(f"\n[full-scale] {info}; peak allocated {peak:.1f} GB; wall {time.perf_counter() - t0:.1f} s")


def need_free(gb):
    free, total = torch.cuda.mem_get_info()
    if free < gb * 1e9:
        pytest.skip(f"needs {gb} GB of free device memory, {free / 1e9:.1f} GB free of {total / 1e9:.1f} GB")
    return f"{free / 1e9:.1f} GB free ({torch.cuda.memory_allocated() / 1e9:.1f} GB held by this process)"


def _field_trainer(model, kind="sgd", weight_decay=0.0):
    """Trainer + FusedRowOptimizer (lr LR; SGD on the bias) as bench.py builds them"""
    from deeplearningrecommendationsystem_b200.optim import FusedRowOptimizer
    from deeplearningrecommendationsystem_b200.trainer import Trainer
    dense = torch.optim.SGD([model.bias], lr=LR) if model.bias.requires_grad else None
    return Trainer(model, torch.nn.BCELoss(), FusedRowOptimizer(model, dense, lr=LR, kind=kind, weight_decay=weight_decay))


# Device memory each case needs: the table, the step's own buffers (FFM: 2.8 GB Jacobian stash), the sparse reference
# (three float64 arrays over the ~0.53 M touched rows: 5.3 GB for FFM) and the guard-row snapshot (1.9 M rows, 3.2 GB
# for FFM).  Peak allocated on a B200, uniform ids: 72.2 GB (FFM), 4.9 GB (FM), 54.5 GB (MF).
FFM_GB, FM_GB, MF_GB = 80, 12, 60


@pytest.mark.gpu
@pytest.mark.parametrize("recompute", ["0", "1"])
@pytest.mark.parametrize("dist", ["uniform", "zipf"])
def test_c2_ffm_full_scale(dist, recompute, big_case, monkeypatch):
    """FieldFFM(C2_CARDS, 16): 56 GB table, B = 65536, lr 0.05.  RS_FFM_RECOMPUTE=0: rs_ffm_fwd (stash) + the streaming
    segment update; =1: the stash-free step, whose once-looked-up rows of the big fields are updated in place by
    ffm_single_kernel."""
    from deeplearningrecommendationsystem_b200.nfield import FieldFFM
    free = need_free(FFM_GB)
    monkeypatch.setenv("RS_FFM_RECOMPUTE", recompute)
    ids, y = make_batch(C2_CARDS, dist, seed=11 if dist == "uniform" else 12)
    m = big_case["model"] = FieldFFM(C2_CARDS, D, fused=True, seed=2, device="cuda")
    tr = big_case["trainer"] = _field_trainer(m)
    assert m._recompute == (recompute == "1")
    keys = ids + torch.tensor(m.offsets_host, device="cuda")
    info = run_steps("ffm", m, tr, (ids,), y.view(-1, 1), keys, m.width, D)
    big_case["info"] = f"ffm {dist} recompute={recompute}: {free}, {info}"


@pytest.mark.gpu
@pytest.mark.parametrize("dist", ["uniform", "zipf"])
def test_c2_fm_full_scale(dist, big_case):
    """FieldFM(C2_CARDS, 16): 33.8 M rows of 16 floats, B = 65536, lr 0.05."""
    from deeplearningrecommendationsystem_b200.nfield import FieldFM
    free = need_free(FM_GB)
    ids, y = make_batch(C2_CARDS, dist, seed=21 if dist == "uniform" else 22)
    m = big_case["model"] = FieldFM(C2_CARDS, D, fused=True, seed=1, device="cuda")
    tr = big_case["trainer"] = _field_trainer(m)
    keys = ids + torch.tensor(m.offsets_host, device="cuda")
    info = run_steps("fm", m, tr, (ids,), y.view(-1, 1), keys, m.width, D)
    big_case["info"] = f"fm {dist}: {free}, {info}"


@pytest.mark.gpu
@pytest.mark.parametrize("dist", ["uniform", "zipf"])
def test_c5_mf_full_scale(dist, big_case):
    """FieldMF(1e8, 1e8, 64): two 100 M-row tables in one 51 GB buffer, B = 65536, lr 0.05."""
    from deeplearningrecommendationsystem_b200.nfield import FieldMF
    free = need_free(MF_GB)
    ids, y = make_batch([C5_ROWS, C5_ROWS], dist, seed=31 if dist == "uniform" else 32)
    m = big_case["model"] = FieldMF(C5_ROWS, C5_ROWS, 64, fused=True, seed=3, device="cuda")
    tr = big_case["trainer"] = _field_trainer(m)
    keys = ids + torch.tensor(m.offsets_host, device="cuda")
    info = run_steps("mf", m, tr, (ids[:, 0].contiguous(), ids[:, 1].contiguous()), y, keys, m.width, None)
    big_case["info"] = f"mf {dist}: {free}, {info}"
