"""DIEN's interest extractor and auxiliary loss (DIEN(..., extractor=True, aux_weight=...)).

  * rs_dien_negatives against `negatives` below, a numpy restatement of the draw with oracle.sampling.philox4x32_10;
    it is itself pinned to rs_sample_negatives' stream (oracle.sampling.negative_draws_philox) on the CPU.
  * rs_dien_aux_fwd / rs_dien_aux_bwd against `aux64`, a float64 restatement, on strided inputs, with g != 1 and
    extreme logits, under a constituent-mass bound; the loss is bit-reproducible.
  * rs_gru_bwd (plain GRU) driven by a per-step gradient g_h_all, the path the extractor's backward takes.
  * model.DIEN(extractor=True) against a float64 autograd restatement built from its state dict, fused rows, the
    ablation aux_weight = 0, eval forwards, the default model.
  * The C4 shape (1 M items, B = 8192, L = 100, D = 64, fused rows, SGD, AUGRU, aux_weight = 1) against the float64
    step reference of test_c3_c4_shapes_gpu plus an auxiliary-loss reference restated here, and graph replay against
    eager.
The restatements and the option checks run without a GPU.
"""
import gc

import numpy as np
import pytest
import torch

from oracle import interactions as OI
from oracle.sampling import negative_draws_philox, philox4x32_10
from test_augru_gpu import _augru_all, _gru_weights, augru, close
from test_c3_c4_shapes_gpu import (C4_B, C4_D, C4_GB, C4_ITEMS, C4_L, C4_LR, DENSE_EPS, _din_unit, _fc, _worst_ratio, c4_batch,
                                   reference)
from test_full_scale_gpu import EPS32, assert_rows_match, big_case, need_free  # noqa: F401

gpu = pytest.mark.gpu


# ---------------------------------------------------------------------------------------------- restatements
def negatives(hist, num_items, seed, epoch, max_blocks=1 << 14):
    """rs_dien_negatives in numpy: slot s = b (L-1) + t, Philox4x32-10 with key = seed and counter = (s lo, s hi, attempt
    block, epoch), candidate (u32 num_items) >> 32, the first of the block's four candidates != hist[b, t+1] wins."""
    hist = np.asarray(hist, dtype=np.int64)
    B, L = hist.shape
    pos = np.clip(hist[:, 1:], 0, num_items - 1).reshape(-1)
    n = pos.size
    out = np.full(n, -1, dtype=np.int64)
    key = np.array([seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF], dtype=np.uint32)
    s = np.arange(n, dtype=np.uint64)
    pending = np.arange(n)
    for blk in range(max_blocks):
        if pending.size == 0:
            break
        sp = s[pending]
        ctr = np.stack([sp & np.uint64(0xFFFFFFFF), sp >> np.uint64(32), np.full(sp.size, blk, np.uint64),
                        np.full(sp.size, epoch & 0xFFFFFFFF, np.uint64)], axis=-1).astype(np.uint32)
        cand = ((philox4x32_10(ctr, key).astype(np.uint64) * np.uint64(num_items)) >> np.uint64(32)).astype(np.int64)
        for j in (3, 2, 1, 0):                  # the first accepted candidate wins: assign in reverse order
            ok = cand[:, j] != pos[pending]
            out[pending[ok]] = cand[ok, j]
        pending = pending[out[pending] < 0]
    return out.reshape(B, L - 1)


def softplus64(x):
    return torch.clamp(x, min=0) + torch.log1p(torch.exp(-x.abs()))


def aux64(h, pos, neg):
    """L_aux in h's dtype: mean over (b, t < L-1) of softplus(-<h_t, pos_t>) + softplus(<h_t, neg_t>); 0 when L = 1"""
    L = h.shape[1]
    if L == 1:
        return h.sum() * 0
    xp, xn = (h[:, :-1] * pos).sum(-1), (h[:, :-1] * neg).sum(-1)
    return (softplus64(-xp) + softplus64(xn)).mean()


# ---------------------------------------------------------------------------------------------- CPU
def test_dien_extractor_options():
    from deeplearningrecommendationsystem_b200 import model as M
    for kw in (dict(aux_weight=1.0), dict(aux_weight=0.0), dict(extractor=True, aux_weight=-0.5),
               dict(extractor=True, aux_weight=float("nan")), dict(extractor=True, aux_weight=float("inf"))):
        with pytest.raises(ValueError):
            M.DIEN(10, 16, **kw)
    with pytest.raises(ValueError):
        M.DIEN(1, 16, extractor=True)
    assert M.DIEN(1, 16, extractor=True, aux_weight=0).aux_weight == 0.0       # the ablation needs no negative
    assert M.DIEN(10, 16, extractor=True).aux_weight == 1.0
    assert M.DIEN(10, 16, extractor=True, aux_weight=0.5).aux_weight == 0.5


def test_dien_extractor_state_dict():
    """extractor=False is today's model; extractor=True adds exactly the four interest_extractor keys, and the seed
    comes from torch's global generator"""
    from deeplearningrecommendationsystem_b200 import model as M
    torch.manual_seed(0)
    a = M.DIEN(10, 16)
    torch.manual_seed(0)
    b = M.DIEN(10, 16, extractor=False)
    torch.manual_seed(0)
    c = M.DIEN(10, 16, evolution="augru", extractor=True)
    sa, sb, sc = a.state_dict(), b.state_dict(), c.state_dict()
    assert list(sa) == list(sb) and all(torch.equal(sa[k], sb[k]) for k in sa)
    assert [n for n, _ in a.named_buffers()] == []
    assert set(sc) - set(sa) == {f"interest_extractor.{w}_{k}_l0" for w in ("weight", "bias") for k in ("ih", "hh")}
    assert set(sa) <= set(sc) and all(torch.equal(sa[k], sc[k]) for k in sa)
    torch.manual_seed(0)
    assert M.DIEN(10, 16, extractor=True).aux_seed == c.aux_seed
    torch.manual_seed(1)
    assert M.DIEN(10, 16, extractor=True).aux_seed != c.aux_seed
    assert int(c.aux_epoch) == 0 and "aux_epoch" not in sc


def test_aux_restatement_matches_the_direct_formula():
    """aux64 (stable softplus) against -log sigmoid(x+) - log(1 - sigmoid(x-)) written out, at |x| up to 200"""
    g = torch.Generator().manual_seed(2)
    B, L, D = 13, 9, 16
    h = torch.randn(B, L, D, generator=g, dtype=torch.float64)
    pos, neg = torch.randn(B, L - 1, D, generator=g, dtype=torch.float64), torch.randn(B, L - 1, D, generator=g, dtype=torch.float64)
    h = h * torch.tensor([0.1, 1.0, 10.0, 40.0], dtype=torch.float64).repeat(4)[:B].view(B, 1, 1)
    xp, xn = (h[:, :-1] * pos).sum(-1), (h[:, :-1] * neg).sum(-1)
    assert float(torch.cat([xp, xn]).abs().max()) > 100
    h[0, 0], pos[0, 0], neg[0, 0] = 0, 0, 0
    h[1, 0, 0], pos[1, 0, 0], neg[1, 0, 0] = 10.0, 20.0, -20.0        # x+ = 200, x- = -200
    h[1, 0, 1:] = 0
    got = aux64(h, pos, neg)
    xp, xn = (h[:, :-1] * pos).sum(-1), (h[:, :-1] * neg).sum(-1)
    want = (torch.log1p(torch.exp(-xp)) + torch.log1p(torch.exp(xn))).sum() / (B * (L - 1))
    assert torch.isfinite(got) and float(softplus64(torch.tensor([-200.0, 200.0], dtype=torch.float64))[1]) == 200.0
    np.testing.assert_allclose(float(got), float(want), rtol=1e-12)
    assert float(aux64(h[:, :1], pos[:, :0], neg[:, :0])) == 0.0


def test_negative_stream_is_rs_sample_negatives_stream():
    """negatives() is oracle.sampling.negative_draws_philox with one user per slot s and (s, hist[b, t+1]) excluded"""
    g = np.random.default_rng(4)
    for num_items, B, L, seed, epoch in ((2, 5, 7, 11, 0), (3, 4, 9, 2 ** 40 + 5, 3), (1000, 6, 5, 77, 2 ** 33 + 1)):
        hist = g.integers(0, num_items, size=(B, L))
        got = negatives(hist, num_items, seed, epoch)
        excl = {(s, int(p)) for s, p in enumerate(hist[:, 1:].reshape(-1))}
        _, want = negative_draws_philox(B * (L - 1), num_items, excl, 1, seed, epoch & 0xFFFFFFFF)
        assert np.array_equal(got.reshape(-1), want)
        assert (got != hist[:, 1:]).all() and (got >= 0).all() and (got < num_items).all()


# ---------------------------------------------------------------------------------------------- negative draw
@gpu
@pytest.mark.parametrize("L", [1, 2, 100])
@pytest.mark.parametrize("num_items", [2, 3, 10 ** 6])
def test_dien_negatives_match_restatement(num_items, L):
    from deeplearningrecommendationsystem_b200 import ops
    g = torch.Generator().manual_seed(num_items + L)
    B, seed = 37, 0x1234_5678_9ABC_DEF0 + L
    hist = torch.randint(0, num_items, (B, L), generator=g)
    draws = []
    for epoch in (0, 1, 5, 2 ** 32 + 1):
        ep = torch.tensor(epoch, dtype=torch.int64, device="cuda")
        got = ops.dien_negatives(hist.cuda(), num_items, seed, ep).cpu()
        assert got.shape == (B, L - 1) and int(ep) == epoch
        assert np.array_equal(got.numpy(), negatives(hist.numpy(), num_items, seed, epoch)), f"epoch {epoch}"
        assert bool((got != hist[:, 1:]).all()) and bool((got >= 0).all()) and bool((got < num_items).all())
        draws.append(got)
    ops.check_status()
    if num_items > 2 and L > 1:
        assert not torch.equal(draws[0], draws[1]), "advancing the epoch did not change the draw"
    assert torch.equal(draws[1], draws[3]), "the epoch enters the counter as 32 bits"


@gpu
def test_dien_negatives_uniform_and_clamped():
    """chi-square over 1000 items (positives uniform, so the draws are too); an out-of-range history id is clamped
    and raises IndexError at the next status check, as a lookup does"""
    from scipy.stats import chisquare
    from deeplearningrecommendationsystem_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(3)
    n = 1000
    hist = torch.randint(0, n, (2000, 51), generator=g, device="cuda")
    neg = ops.dien_negatives(hist, n, 99, torch.zeros((), dtype=torch.int64, device="cuda"))
    counts = torch.bincount(neg.view(-1), minlength=n).cpu().numpy()
    assert chisquare(counts).pvalue > 1e-4
    ops.check_status()
    bad = hist[:2, :3].clone()
    bad[0, 1] = n + 7
    got = ops.dien_negatives(bad, n, 99, torch.zeros((), dtype=torch.int64, device="cuda"))
    assert int(got[0, 0]) != n - 1 and int(got[0, 0]) < n
    with pytest.raises(IndexError):
        ops.check_status()


# ---------------------------------------------------------------------------------------------- aux kernels
def _aux_case(g, B, L, D):
    """strided float64 operands: h a slice of a wider buffer, pos / neg slices of one (B, 2L, D) row block; per-sample
    scales 0.1 .. 40 put the logits of some samples far into the tails"""
    wide = torch.randn(B, L + 3, D, generator=g, dtype=torch.float64)
    scale = torch.tensor([0.1, 1.0, 3.0, 40.0], dtype=torch.float64).repeat(B)[:B].view(B, 1, 1)
    rows = torch.randn(B, 2 * L, D, generator=g, dtype=torch.float64)
    return (wide * scale)[:, 1:L + 1], rows, rows[:, 1:L], rows[:, L + 1:]


@gpu
@pytest.mark.parametrize("L", [1, 2, 3, 100])
@pytest.mark.parametrize("D", [16, 32, 64])
def test_dien_aux_kernels_match_float64(D, L):
    from deeplearningrecommendationsystem_b200 import ops
    g = torch.Generator().manual_seed(D * 1000 + L)
    B = 37
    h64, rows64, pos64, neg64 = _aux_case(g, B, L, D)
    # fp32 operands on the device with the same strides: h inside its wider buffer, pos / neg inside the row block
    wide = torch.zeros(B, L + 3, D, device="cuda")
    wide[:, 1:L + 1] = h64.float().cuda()
    h, rows = wide[:, 1:L + 1], rows64.float().cuda()
    pos, neg = rows[:, 1:L], rows[:, L + 1:]
    assert not h.is_contiguous() or L == 1
    h64, pos64, neg64 = (t.float().double() for t in (h64, pos64, neg64))      # the fp32 values themselves
    loss, sig = ops.dien_aux_fwd(h, pos, neg)
    assert sig.shape == (B, L - 1, 2)
    loss2, sig2 = ops.dien_aux_fwd(h, pos, neg)
    assert torch.equal(loss, loss2) and torch.equal(sig, sig2), "the forward is not reproducible"
    want = aux64(h64, pos64, neg64)
    xp, xn = (h64[:, :-1] * pos64).sum(-1), (h64[:, :-1] * neg64).sum(-1)
    Mp, Mn = (h64[:, :-1].abs() * pos64.abs()).sum(-1), (h64[:, :-1].abs() * neg64.abs()).sum(-1)
    if L > 1:
        assert float(torch.cat([xp, xn]).abs().max()) > 100, "no extreme logits in the case"
    # loss: each softplus has slope <= 1, so its error is the dot product's: a 4-term fma chain per lane and a
    # log2(D/4)-level shuffle tree, <= 8 eps32 of the dot's mass
    bound = 1e-5 * abs(float(want)) + 8 * EPS32 * float((Mp + Mn).mean() if L > 1 else 0.0)
    assert abs(float(loss) - float(want)) <= bound, (float(loss), float(want), bound)
    assert bool(torch.isfinite(loss)) and bool(torch.isfinite(sig).all())
    s0, s1 = -torch.sigmoid(-xp), torch.sigmoid(xn)
    e0 = 1e-6 * s0.abs() + s0.abs() * (1 + s0) * 8 * EPS32 * Mp + 1e-30            # |d sig / d x| (8 eps32 M) + rounding
    e1 = 1e-6 * s1.abs() + s1 * (1 - s1) * 8 * EPS32 * Mn + 1e-30
    sg = sig.cpu().double()
    assert bool(((sg[..., 0] - s0).abs() <= e0).all()) and bool(((sg[..., 1] - s1).abs() <= e1).all()), "sig off float64"
    # backward with g != 1 read from the device
    gval = torch.tensor(0.37, device="cuda")
    dh, dp, dn = ops.dien_aux_bwd(h, pos, neg, sig, gval)
    again = ops.dien_aux_bwd(h, pos, neg, sig, gval)
    assert all(torch.equal(a, b) for a, b in zip((dh, dp, dn), again)), "the backward is not reproducible"
    assert not bool(dh[:, -1].any()), "dh of the last state must be zero"
    hh, pp, nn_ = (t.clone().requires_grad_(True) for t in (h64, pos64, neg64))
    gr = torch.autograd.grad(aux64(hh, pp, nn_) * float(gval), [hh, pp, nn_], allow_unused=True)
    gr = [torch.zeros_like(t) if x is None else x for x, t in zip(gr, (hh, pp, nn_))]
    if L == 1:
        assert not bool(dh.any()) and dp.numel() == 0 and dn.numel() == 0
        return
    c = float(gval) / (B * (L - 1))
    # constituent mass: c [ (|s0| e|.| + e0 |.|) terms ] -- the error of each stashed derivative times its operand, plus a
    # few eps32 of the products themselves
    m_h = c * ((s0.abs().unsqueeze(-1) * pos64.abs() + s1.unsqueeze(-1) * neg64.abs()) * 4 * EPS32
               + e0.unsqueeze(-1) * pos64.abs() + e1.unsqueeze(-1) * neg64.abs())
    m_p = c * (s0.abs().unsqueeze(-1) * 2 * EPS32 + e0.unsqueeze(-1)) * h64[:, :-1].abs()
    m_n = c * (s1.unsqueeze(-1) * 2 * EPS32 + e1.unsqueeze(-1)) * h64[:, :-1].abs()
    for name, got_, want_, m in (("dh", dh[:, :-1], gr[0][:, :-1], m_h), ("d_pos", dp, gr[1], m_p), ("d_neg", dn, gr[2], m_n)):
        err = (got_.cpu().double() - want_).abs()
        bnd = 1e-6 * want_.abs() + m + 1e-38
        assert bool((err <= bnd).all()), f"{name}: off float64 by {_worst_ratio(err, bnd):.2f} of the bound"


@gpu
def test_dien_aux_kernel_limits():
    from deeplearningrecommendationsystem_b200 import ops
    h = torch.zeros(4, 5, 48, device="cuda")
    with pytest.raises(RuntimeError, match="16, 32, 64"):
        ops.dien_aux_fwd(h, h[:, 1:], h[:, 1:])
    e = torch.zeros(0, 5, 16, device="cuda")
    loss, sig = ops.dien_aux_fwd(e, e[:, 1:], e[:, 1:])
    assert float(loss) == 0.0 and sig.shape == (0, 4, 2)
    dh, dp, dn = ops.dien_aux_bwd(e, e[:, 1:], e[:, 1:], sig, torch.ones((), device="cuda"))
    assert dh.shape == (0, 5, 16) and dp.shape == (0, 4, 16)


# ---------------------------------------------------------------------------------------------- plain GRU, g_h_all
@gpu
@pytest.mark.parametrize("with_last", [False, True])
@pytest.mark.parametrize("H,B,L", [(8, 17, 3), (16, 50, 1), (32, 33, 40), (64, 21, 100)])
def test_gru_bwd_per_step_gradient_matches_float64(H, B, L, with_last):
    """rs_gru_bwd (the plain GRU) from g_h_all alone and from g_h_all + g_h_last, against autograd of the float64
    recurrence (_augru_all with att == 1 is the GRU)"""
    from deeplearningrecommendationsystem_b200 import ops
    g = torch.Generator().manual_seed(11 * H + L)
    _, w_hh, _, b_hh = _gru_weights(g, 3 * H, H)
    gi = (torch.randn(B, L, 3 * H, generator=g, dtype=torch.float64) * 0.7).requires_grad_(True)
    w_hh, b_hh = w_hh.requires_grad_(True), b_hh.requires_grad_(True)
    want = _augru_all(gi, torch.ones(B, L, dtype=torch.float64), w_hh, b_hh)
    g_all, g_last = torch.randn(B, L, H, generator=g, dtype=torch.float64), torch.randn(B, H, generator=g, dtype=torch.float64)
    obj = (want * g_all).sum() + ((want[:, -1] * g_last).sum() if with_last else 0)
    grads = torch.autograd.grad(obj, [gi, w_hh, b_hh])
    c32 = lambda t: t.detach().float().cuda()              # noqa: E731
    h_all, gates = ops.gru_fwd(c32(gi), c32(w_hh), c32(b_hh))
    close(h_all, want, msg="h_all")
    d_gi, d_gh = ops.gru_bwd(c32(w_hh), h_all, gates, g_h_all=c32(g_all), g_h_last=c32(g_last) if with_last else None)
    h_prev = torch.cat([torch.zeros(B, 1, H), h_all.cpu()[:, :-1]], dim=1).double()
    d_gh64 = d_gh.cpu().double().reshape(-1, 3 * H)
    got = {"d_gi": d_gi, "dW_hh (d_gh)": d_gh64.t() @ h_prev.reshape(-1, H), "db_hh (d_gh)": d_gh64.sum(0)}
    for (name, a), w_ in zip(got.items(), grads):
        close(a, w_, rtol=1e-5, atol=2e-6 * max(1.0, float(w_.abs().max())), msg=name)
    r = gates.view(B, L, 4, H)[:, :, 0]
    assert torch.equal(d_gh[..., :2 * H], d_gi[..., :2 * H]) and torch.equal(d_gh[..., 2 * H:], d_gi[..., 2 * H:] * r)


@gpu
def test_gru_sequence_matches_nn_gru():
    """attention.gru_sequence: nn.GRU's output and its gradients (every h_t gets an upstream gradient), nn.GRU run in
    float64 on the CPU (on the GPU it is cuDNN, which may take TF32)"""
    from deeplearningrecommendationsystem_b200 import attention
    g = torch.Generator().manual_seed(5)
    gru = torch.nn.GRU(32, 32, batch_first=True)
    x = torch.randn(40, 9, 32, generator=g) * 0.5
    gup = torch.randn(40, 9, 32, generator=g)
    gru64, x64 = torch.nn.GRU(32, 32, batch_first=True).double(), x.double().requires_grad_(True)
    gru64.load_state_dict({k: v.double() for k, v in gru.state_dict().items()})
    ref = gru64(x64)[0]
    want = torch.autograd.grad((ref * gup.double()).sum(), [x64] + list(gru64.parameters()))
    gru, x = gru.cuda(), x.cuda().requires_grad_(True)
    out = attention.gru_sequence(x, gru)
    got = torch.autograd.grad((out * gup.cuda()).sum(), [x] + list(gru.parameters()))
    close(out, ref, atol=1e-6)
    for a, b in zip(got, want):
        close(a, b, rtol=1e-4, atol=1e-5 * max(1.0, float(b.abs().max())))


# ---------------------------------------------------------------------------------------------- the model
SMALL = dict(items=300, D=16, L=7, B=200)


def _small_model(evolution, aux_weight, seed=0):
    from deeplearningrecommendationsystem_b200 import model as M
    torch.manual_seed(seed)
    m = M.DIEN(SMALL["items"], SMALL["D"], evolution=evolution, extractor=True, aux_weight=aux_weight)
    with torch.no_grad():                      # biases away from zero: the ReLU masks are not all-or-nothing
        for n, p in m.named_parameters():
            if n.endswith("bias"):
                p.normal_(0.0, 0.2)
    return m


def _small_batch(seed):
    g = torch.Generator().manual_seed(seed)
    hist = torch.randint(0, SMALL["items"], (SMALL["B"], SMALL["L"]), generator=g)
    tgt = torch.randint(0, SMALL["items"], (SMALL["B"],), generator=g)
    return hist, tgt, (torch.rand(SMALL["B"], 1, generator=g) < 0.4).float()


def _gru_w(sd, pfx):
    return [sd[f"{pfx}.{k}"] for k in ("weight_ih_l0", "weight_hh_l0", "bias_ih_l0", "bias_hh_l0")]


def dien_x64(sd, hist, tgt, neg, evolution, aux_weight):
    """model.DIEN(extractor=True) restated from its state dict (oracle.interactions, augru, _augru_all) in sd's dtype
    -> (pred (B,), aux_weight * L_aux)"""
    tab = sd["din.item_embedding.weight"]
    e, t = tab[hist], tab[tgt]
    w_ih, w_hh, b_ih, b_hh = _gru_w(sd, "interest_extractor")
    hs = _augru_all(e @ w_ih.t() + b_ih, torch.ones(hist.shape, dtype=e.dtype), w_hh, b_hh)      # att == 1: the GRU
    att = OI.din_attention(hs, t, [(sd[f"din.attention.{k}.weight"], sd[f"din.attention.{k}.bias"]) for k in (0, 2, 4)])
    ev = _gru_w(sd, "interest_evolution")
    hL = augru(hs, att, *ev) if evolution == "augru" else OI.gru(hs * att.unsqueeze(-1), *ev)
    f = OI.relu_tower(torch.cat([hL, t], dim=1), [(sd[f"fc.{k}.weight"], sd[f"fc.{k}.bias"]) for k in (0, 2, 4)], relu_last=False)
    aux = aux64(hs, tab[hist[:, 1:]], tab[neg]) * aux_weight if aux_weight > 0 else None
    return torch.sigmoid(f).view(-1), aux


@gpu
@pytest.mark.parametrize("aux_weight", [0.0, 0.5, 1.0])
@pytest.mark.parametrize("evolution", ["gru", "augru"])
def test_small_dien_extractor_matches_float64(evolution, aux_weight, monkeypatch):
    """predictions, BCE, model.aux_loss and every gradient (interest_extractor included) against autograd of the
    float64 restatement with negatives from the restated stream; then two torch-Adam steps.  aux_weight = 0 draws
    nothing and runs no auxiliary kernel; eval and no_grad forwards leave the epoch alone."""
    from deeplearningrecommendationsystem_b200 import ops
    m = _small_model(evolution, aux_weight)
    sd64 = {k: v.detach().double().clone().requires_grad_(True) for k, v in m.state_dict().items()}
    m = m.cuda()
    if aux_weight == 0:
        def refuse(*a, **kw):
            raise AssertionError("aux_weight = 0 ran an auxiliary-loss op")
        for name in ("dien_negatives", "dien_aux_fwd", "dien_aux_bwd"):
            monkeypatch.setattr(ops, name, refuse)
    hist, tgt, y = _small_batch(1)
    lr = 1e-3
    opt = torch.optim.Adam(m.parameters(), lr=lr)
    opt64 = torch.optim.Adam(list(sd64.values()), lr=lr)
    names = [n for n, _ in m.named_parameters()]
    assert any(n.startswith("interest_extractor.") for n in names)
    first = None
    for step in range(2):
        assert int(m.aux_epoch) == (step if aux_weight > 0 else 0)
        neg = torch.from_numpy(negatives(hist.numpy(), SMALL["items"], m.aux_seed, step))
        opt.zero_grad()
        opt64.zero_grad()
        p = m(hist.cuda(), tgt.cuda())
        loss = torch.nn.BCELoss()(p, y.cuda())
        loss.backward()
        p64, aux64_ = dien_x64(sd64, hist, tgt, neg, evolution, aux_weight)
        loss64 = OI.bce(p64, y.view(-1).double())
        (loss64 + (aux64_ if aux64_ is not None else 0)).backward()
        close(p.view(-1), p64, msg=f"step {step} pred")
        close(loss, loss64, msg=f"step {step} BCE")
        if aux_weight > 0:
            close(m.aux_loss, aux64_, msg=f"step {step} aux_loss")
        else:
            assert m.aux_loss is None
        for n, q in m.named_parameters():
            g64 = sd64[n].grad
            tol = 1e-5 * float(g64.abs().max())
            if n == "din.attention.4.bias":        # softmax is shift invariant: analytically zero, both sides are noise
                tol = 1e-5 * float(sd64["din.attention.4.weight"].grad.abs().max())
            close(q.grad, g64, rtol=1e-5, atol=max(tol, 1e-9), msg=f"step {step} {n}.grad")
        if first is None:
            first = {n: sd64[n].grad.abs() for n in names}
        opt.step()
        opt64.step()
    for n, q in m.named_parameters():
        settled = first[n] > 1e-2 * float(first[n].max())
        err = (q.detach().cpu().double() - sd64[n].detach()).abs()
        if bool(settled.any()):
            assert float(err[settled].max()) <= 1e-3 * lr + 1e-6 * float(sd64[n].detach().abs().max()), n
        assert float(err.max()) <= 4 * lr, n
    # eval and no_grad forwards: no draw, the epoch stays; the prediction is the training forward's
    ep = int(m.aux_epoch)
    with torch.no_grad():
        p_ng = m(hist.cuda(), tgt.cuda())
    m.eval()
    p_ev = m(hist.cuda(), tgt.cuda())
    m.train()
    assert int(m.aux_epoch) == ep and torch.equal(p_ng, p_ev.detach())
    m.recommendation(2, SMALL["items"], hist[:2].tolist(), 5)
    assert int(m.aux_epoch) == ep


@gpu
def test_small_dien_extractor_fused_rows_and_default():
    """fused sparse rows with SGD give the parameters of SGD on dense tables (negatives included); the default DIEN
    is bit-identical to extractor=False"""
    from deeplearningrecommendationsystem_b200 import model as M
    from deeplearningrecommendationsystem_b200.optim import FusedRowOptimizer
    from deeplearningrecommendationsystem_b200.trainer import Trainer
    lr = 0.05
    dense, fused = _small_model("augru", 1.0).cuda(), _small_model("augru", 1.0).cuda().fuse_embedding_updates()
    assert dense.aux_seed == fused.aux_seed
    tr_d = Trainer(dense, torch.nn.BCELoss(), torch.optim.SGD(dense.parameters(), lr=lr))
    tr_f = Trainer(fused, torch.nn.BCELoss(), FusedRowOptimizer(fused, torch.optim.SGD(
        [p for p in fused.parameters() if p.requires_grad], lr=lr), lr=lr, kind="sgd"))
    for step in range(2):
        hist, tgt, y = _small_batch(10 + step)
        tr_d.train_loop(hist.cuda(), tgt.cuda(), train_rating=y.cuda())
        tr_f.train_loop(hist.cuda(), tgt.cuda(), train_rating=y.cuda())
        close(tr_f.predictions_train, tr_d.predictions_train, msg=f"step {step} pred")
        close(fused.aux_loss, dense.aux_loss, msg=f"step {step} aux_loss")
        close(tr_f.train_loss, tr_d.train_loss, msg=f"step {step} train_loss")
    assert int(dense.aux_epoch) == int(fused.aux_epoch) == 2
    for (n, a), (_, b) in zip(dense.state_dict().items(), fused.state_dict().items()):
        close(b, a, rtol=1e-5, atol=1e-6, msg=n)
    hist, tgt, y = (t.cuda() for t in _small_batch(20))
    outs = []
    for kw in ({}, {"extractor": False}):
        torch.manual_seed(5)
        m = M.DIEN(SMALL["items"], SMALL["D"], **kw).cuda()
        p = m(hist, tgt)
        torch.nn.BCELoss()(p, y).backward()
        outs.append([p.detach()] + [q.grad.clone() for q in m.parameters()])
    assert all(torch.equal(u, v) for u, v in zip(*outs)), "extractor=False differs from the default"


# ---------------------------------------------------------------------------------------------- the C4 shape
def _states(gi, Whh, bhh, att, am, tr, key):
    """every h_t of the AUGRU (att (c, L); att == 1 is the GRU) on projections gi (c, L, 3H).  In the mass pass the
    gates and weights keep their real values and pass on the magnitude of their derivative (dien_augru_logit's rule)."""
    H = Whh.shape[1]
    hs, out = gi.new_zeros(gi.shape[0], H), []
    for s in range(gi.shape[1]):
        gh = hs @ Whh.t() + bhh
        xr, xz = gi[:, s, :H] + gh[:, :H], gi[:, s, H:2 * H] + gh[:, H:2 * H]
        a = att[:, s:s + 1]
        if not am:
            r, z = torch.sigmoid(xr), torch.sigmoid(xz)
            n = torch.tanh(gi[:, s, 2 * H:] + r * gh[:, 2 * H:])
            tr[(key, s)] = (r.detach(), z.detach(), n.detach())
            u = a * (1.0 - z)
            hs = (1.0 - u) * hs + u * n
        else:
            r0, z0, n0 = tr[(key, s)]
            r = r0 + r0 * (1 - r0) * (xr - xr.detach())
            z = z0 + z0 * (1 - z0) * (xz - xz.detach())
            xn = gi[:, s, 2 * H:] + r * gh[:, 2 * H:]
            n = n0.abs() + (1 - n0 * n0) * (xn - xn.detach())
            a0 = a.detach()
            u0 = a0 * (1 - z0)
            du = (1 - z0) * (a - a0) + a0 * (z - z.detach())
            hs = (1.0 - u0) * hs + u0 * n + du * (n.detach() + hs.detach())
        out.append(hs)
    return torch.stack(out, dim=1)


def _extract(P, X, L, am, tr):
    ones = X.new_ones(X.shape[0], L)
    gi = X[:, :L] @ P["interest_extractor.weight_ih_l0"].t() + P["interest_extractor.bias_ih_l0"]
    return _states(gi, P["interest_extractor.weight_hh_l0"], P["interest_extractor.bias_hh_l0"], ones, am, tr, "x")


def dien_x_logit(P, X, M, am, tr):
    """model.DIEN(evolution="augru", extractor=True) for the step reference: X (c, 2L, D) = [history | target |
    negatives] rows (the negatives only enter the auxiliary term, see aux_reference)"""
    checks = []
    L = X.shape[1] // 2
    hs = _extract(P, X, L, am, tr)
    att_rows = torch.cat([hs, X[:, L:L + 1]], dim=1)
    w = _din_unit(P, att_rows, M, am, tr, "din.", checks)
    gi = hs @ P["interest_evolution.weight_ih_l0"].t() + P["interest_evolution.bias_ih_l0"]
    hL = _states(gi, P["interest_evolution.weight_hh_l0"], P["interest_evolution.bias_hh_l0"], w, am, tr, "e")[:, -1]
    return _fc(P, torch.cat([hL, X[:, L]], dim=1), M, am, checks), checks


def aux_reference(params, rows, inv, aux_weight, chunk):
    """aux_weight * L_aux of one step in float64 and its gradients, chunked like `reference`: value, the gradient and
    constituent mass of every dense parameter (the extractor's; zero elsewhere) and of the rows.  In the mass pass the
    softplus slopes |sigma(x+) - 1|, sigma(x-) are kept and the dot products take |.| operands."""
    nb, K = inv.shape
    L = K // 2
    npairs = nb * (L - 1)
    P = {n: p.detach().double().requires_grad_(True) for n, p in params.items()}
    A = {n: p.detach().double().abs().requires_grad_(True) for n, p in params.items()}
    out = {"aux": torch.zeros((), dtype=torch.float64, device=rows.device),
           "grads": {n: torch.zeros_like(p) for n, p in P.items()}, "mass": {n: torch.zeros_like(p) for n, p in P.items()}}
    g_rows, S = (torch.zeros(rows.shape, dtype=torch.float64, device=rows.device) for _ in range(2))
    keys = [n for n in P if n.startswith("interest_extractor.")]
    for s in range(0, nb, chunk):
        idx = inv[s:s + chunk]
        flat = idx.reshape(-1)
        tr = {}
        X = rows[idx].double().requires_grad_(True)
        hs = _extract(P, X, L, False, tr)[:, :-1]
        xp, xn = (hs * X[:, 1:L]).sum(-1), (hs * X[:, L + 1:]).sum(-1)
        val = (softplus64(-xp) + softplus64(xn)).sum() * (aux_weight / npairs)
        gs = torch.autograd.grad(val, [X] + [P[k] for k in keys])
        g_rows.index_add_(0, flat, gs[0].reshape(flat.numel(), -1))
        for k, gk in zip(keys, gs[1:]):
            out["grads"][k] += gk
        out["aux"] += val.detach()
        s0, s1 = torch.sigmoid(-xp).detach(), torch.sigmoid(xn).detach()
        del X, hs, xp, xn, val, gs
        Xa = rows[idx].double().abs().requires_grad_(True)
        ha = _extract(A, Xa, L, True, tr)[:, :-1]
        va = (s0 * (ha * Xa[:, 1:L]).sum(-1) + s1 * (ha * Xa[:, L + 1:]).sum(-1)).sum() * (aux_weight / npairs)
        ga = torch.autograd.grad(va, [Xa] + [A[k] for k in keys])
        S.index_add_(0, flat, ga[0].reshape(flat.numel(), -1))
        for k, gk in zip(keys, ga[1:]):
            out["mass"][k] += gk
        del Xa, ha, va, ga, tr
    out["g_rows"], out["S"] = g_rows, S
    return out


def test_extractor_step_reference_matches_the_oracle():
    """reference(dien_x_logit) + aux_reference with masks = (z > 0), float64 on the CPU, against autograd of dien_x64:
    predictions, BCE, aux, every dense gradient and the summed row gradient to 1e-12; the mass passes bound them"""
    from deeplearningrecommendationsystem_b200 import model as M
    torch.manual_seed(3)
    items, D, L, nb, w = 60, 8, 7, 200, 0.7
    m = M.DIEN(items, D, evolution="augru", extractor=True, aux_weight=w).double()
    with torch.no_grad():
        for n, p in m.named_parameters():
            if n.endswith("bias"):
                p.normal_(0.0, 0.2)
    sd = {k: v.detach().clone() for k, v in m.state_dict().items()}
    g = torch.Generator().manual_seed(9)
    hist, tgt = torch.randint(0, items, (nb, L), generator=g), torch.randint(0, items, (nb,), generator=g)
    y = (torch.rand(nb, generator=g) < 0.4).double()
    neg = torch.from_numpy(negatives(hist.numpy(), items, m.aux_seed, 0))
    tab = sd["din.item_embedding.weight"]
    ex = _gru_w(sd, "interest_extractor")
    hs = _augru_all(tab[hist] @ ex[0].t() + ex[2], torch.ones(nb, L, dtype=torch.float64), ex[1], ex[3])
    t = tab[tgt]
    x = torch.cat([hs, hs - t.unsqueeze(1), t.unsqueeze(1).expand_as(hs)], dim=-1)
    z0 = x @ sd["din.attention.0.weight"].t() + sd["din.attention.0.bias"]
    z1 = torch.relu(z0) @ sd["din.attention.2.weight"].t() + sd["din.attention.2.bias"]
    att = torch.softmax((torch.relu(z1) @ sd["din.attention.4.weight"].t() + sd["din.attention.4.bias"]).squeeze(-1), dim=-1)
    hL = augru(hs, att, *_gru_w(sd, "interest_evolution"))
    a = torch.cat([hL, t], dim=1) @ sd["fc.0.weight"].t() + sd["fc.0.bias"]
    b = torch.relu(a) @ sd["fc.2.weight"].t() + sd["fc.2.bias"]
    masks = {"act0": z0 > 0, "act1": z1 > 0, "act0_val": torch.relu(z0), "act1_val": torch.relu(z1), "attw_val": att, "fc.1": a > 0,
             "fc.3": b > 0}
    leaves = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    pred, aux = dien_x64(leaves, hist, tgt, neg, "augru", w)
    bce = OI.bce(pred, y)
    params = {k: v for k, v in sd.items() if not k.endswith("item_embedding.weight")}
    got = torch.autograd.grad(bce + aux, [leaves["din.item_embedding.weight"]] + [leaves[k] for k in params])
    keys = torch.cat([hist, tgt.unsqueeze(1), neg], dim=1)
    uniq, inv = torch.unique(keys, return_inverse=True)
    ref = reference(dien_x_logit, params, tab[uniq], inv, y, masks, chunk=70)
    ax = aux_reference(params, tab[uniq], inv, w, chunk=70)
    c = lambda u, v, what: np.testing.assert_allclose(u.detach().numpy(), v.detach().numpy(), rtol=1e-12, atol=1e-15, err_msg=what)  # noqa: E731
    c(ref["pred"], pred, "pred")
    c(ref["loss"], bce, "bce")
    c(ax["aux"], aux, "aux")
    c(ref["g_rows"] + ax["g_rows"], got[0][uniq], "rows")
    for k, gk in zip(params, got[1:]):
        c(ref["grads"][k] + ax["grads"][k], gk, k)
        assert bool((ref["mass"][k] + ax["mass"][k] >= gk.abs() * (1 - 1e-12)).all()), k
    assert bool((ref["S"] + ax["S"] >= got[0][uniq].abs() * (1 - 1e-12)).all())
    assert float(ax["grads"]["interest_extractor.weight_ih_l0"].abs().max()) > 0


def _c4_model(seed=0):
    from deeplearningrecommendationsystem_b200 import model as M
    from deeplearningrecommendationsystem_b200.optim import FusedRowOptimizer
    torch.manual_seed(seed)
    m = M.DIEN(C4_ITEMS, C4_D, evolution="augru", extractor=True, aux_weight=1.0).cuda().fuse_embedding_updates()
    return m, FusedRowOptimizer(m, torch.optim.SGD([p for p in m.parameters() if p.requires_grad], lr=C4_LR), lr=C4_LR, kind="sgd")


@gpu
def test_c4_extractor_step_matches_float64(big_case, monkeypatch):
    """DIEN(1 M items, 64, evolution="augru", extractor=True, aux_weight=1) at B = 8192, L = 100, lr 0.01, fused rows +
    SGD: two steps of Trainer.train_loop against `reference` (BCE, the kernels' ReLU masks) plus aux_reference, with
    negatives from the restated stream; every touched row, every dense gradient and parameter; untouched rows stay
    bit-identical"""
    from deeplearningrecommendationsystem_b200 import ops
    from deeplearningrecommendationsystem_b200.trainer import Trainer
    free = need_free(C4_GB)
    (hist, tgt), y = c4_batch(54)
    m, opt = _c4_model()
    big_case["model"] = m
    tr = big_case["trainer"] = Trainer(m, torch.nn.BCELoss(), opt)
    cap = big_case["capture"] = {}
    real = ops.din_fwd

    def din_fwd(*a, **kw):
        out = real(*a, **kw)
        if kw.get("want_stash"):
            assert out[2] is not None, "the C4 attention unit did not take the tensor-core path"
            cap["stash"] = out[2]
        return out
    monkeypatch.setattr(ops, "din_fwd", din_fwd)
    for k in (1, 3):
        m.fc[k].register_forward_hook(lambda mod, inp, out, k=k: cap.__setitem__(f"fc.{k}", out.detach() > 0))

    def capture():
        attw, act0, act1 = cap["stash"]
        a0, a1 = act0.view(C4_B, C4_L, -1), act1.view(C4_B, C4_L, -1)
        return {"fc.1": cap["fc.1"], "fc.3": cap["fc.3"], "act0": a0 > 0, "act1": a1 > 0, "act0_val": a0, "act1_val": a1, "attw_val": attw}
    table = m.din.item_embedding.weight.data
    params = {n: p for n, p in m.named_parameters() if p.requires_grad and not n.endswith("item_embedding.weight")}
    hist_np = hist.cpu().numpy()
    worst = {"rows": 0.0}
    for step in (1, 2):
        what = f"c4 dien extractor step {step}"
        neg = torch.from_numpy(negatives(hist_np, C4_ITEMS, m.aux_seed, int(m.aux_epoch))).cuda()
        keys = torch.cat([hist, tgt.unsqueeze(1), neg], dim=1)
        uniq, inv = torch.unique(keys, return_inverse=True)
        keep = torch.ones(table.shape[0], dtype=torch.bool, device="cuda")
        keep[uniq] = False
        guard = keep.nonzero().view(-1)
        del keep
        snap = table[guard].view(torch.int32).clone()
        before = table[uniq].clone()
        pbefore = {n: p.detach().clone() for n, p in params.items()}
        tr.train_loop(hist, tgt, train_rating=y)
        ops.check_status()
        ref = reference(dien_x_logit, pbefore, before, inv, y, capture(), 1024)
        ax = aux_reference(pbefore, before, inv, 1.0, 1024)
        np.testing.assert_allclose(tr.predictions_train.detach().reshape(-1).cpu().numpy(), ref["pred"].cpu().numpy(),
                                   rtol=1e-5, atol=1e-6, err_msg=what)
        np.testing.assert_allclose(float(tr.train_loss), float(ref["loss"]), rtol=1e-5, err_msg=what)
        np.testing.assert_allclose(float(m.aux_loss), float(ax["aux"]), rtol=1e-5, err_msg=what)
        g64, S = ref["g_rows"] + ax["g_rows"], ref["S"] + ax["S"]
        rows64 = before.double() - C4_LR * g64
        worst["rows"] = max(worst["rows"], assert_rows_match(table[uniq], {"rows": rows64, "grad": g64, "absg": S}, C4_LR, what))
        del before, rows64, g64, S
        for n, p in params.items():
            g, M_ = ref["grads"][n] + ax["grads"][n], ref["mass"][n] + ax["mass"][n]
            bound = 1e-5 * g.abs() + DENSE_EPS * EPS32 * M_
            if n.endswith("attention.4.bias"):
                bound = bound + 1e-5 * float(ref["grads"][n[:-4] + "weight"].abs().max())
            r = _worst_ratio((p.grad.double() - g).abs(), bound)
            assert r <= 1.0, f"{what}: {n}.grad off float64 by {r:.2f} of the bound"
            want = pbefore[n].double() - C4_LR * g
            pr = _worst_ratio((p.detach().double() - want).abs(), 1e-6 * want.abs() + C4_LR * bound)
            assert pr <= 1.0, f"{what}: updated {n} off float64 by {pr:.2f} of the bound"
            grp = n.split(".")[0]
            worst[grp] = max(worst.get(grp, 0.0), r, pr)
        same = table[guard].view(torch.int32) == snap
        assert bool(same.all()), f"{what}: {int((~same.all(1)).sum())} untouched rows changed"
        del ref, ax, snap, guard, pbefore
    assert int(m.aux_epoch) == 2
    big_case["info"] = f"c4 dien extractor: {free}, worst err/bound " + ", ".join(f"{k} {v:.2e}" for k, v in worst.items())


@gpu
def test_c4_extractor_graphed_step_equals_eager(big_case, monkeypatch):
    """GraphedTrainStep(warmup=1) against eager Trainer.train_loop from the same state and epoch over three steps:
    bit-identical predictions, losses, aux_loss, parameters and tables; every replay draws the restated negatives of
    its own epoch (the third step repeats the second's batch, so only the epoch tells them apart)"""
    from deeplearningrecommendationsystem_b200 import ops
    from deeplearningrecommendationsystem_b200.graph import GraphedTrainStep
    from deeplearningrecommendationsystem_b200.trainer import Trainer
    free = need_free(C4_GB)
    (m1, o1), (m2, o2) = _c4_model(4), _c4_model(4)
    big_case["model"] = (m1, m2)
    assert m1.aux_seed == m2.aux_seed
    tr = Trainer(m1, torch.nn.BCELoss(), o1)
    gs = GraphedTrainStep(m2, torch.nn.BCELoss(), o2, warmup=1)
    drawn = {}                                 # epoch buffer -> the last negatives tensor drawn for that model
    real = ops.dien_negatives

    def dien_negatives(hist, num_items, seed, epoch):
        out = real(hist, num_items, seed, epoch)
        drawn[epoch.data_ptr()] = out
        return out
    monkeypatch.setattr(ops, "dien_negatives", dien_negatives)
    batches = [c4_batch(90), c4_batch(91)]
    batches.append(batches[1])
    for k, (ins, y) in enumerate(batches):
        tr.train_loop(*ins, train_rating=y)
        eager_neg = drawn[m1.aux_epoch.data_ptr()].clone()
        pred, loss = gs(*ins, rating=y)
        graph_neg = drawn[m2.aux_epoch.data_ptr()]     # the warm-up's tensor, then the captured one every replay rewrites
        assert torch.equal(graph_neg, eager_neg), f"step {k}: the graphed step drew other negatives"
        want = negatives(ins[0].cpu().numpy(), C4_ITEMS, m1.aux_seed, k)
        assert np.array_equal(graph_neg.cpu().numpy(), want), f"step {k}: negatives are not the epoch-{k} draw"
        assert torch.equal(pred, tr.predictions_train), f"step {k}: predictions differ"
        assert torch.equal(loss, tr.train_loss), f"step {k}: losses differ"
        assert torch.equal(m2.aux_loss, m1.aux_loss), f"step {k}: aux losses differ"
    assert gs.graph is not None and int(m1.aux_epoch) == int(m2.aux_epoch) == 3
    for (n, a), (_, b) in zip(m1.named_parameters(), m2.named_parameters()):
        assert torch.equal(a, b), f"{n} differs between the graphed and the eager step"
    assert torch.equal(m1.din.item_embedding.weight, m2.din.item_embedding.weight)
    big_case["info"] = f"graphed == eager dien extractor: {free}"
    del gs, tr
    gc.collect()
