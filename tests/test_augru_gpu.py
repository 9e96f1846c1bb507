"""DIEN's attention-gated GRU (AUGRU) and the attention-weights mode of the DIN attention unit.

  * rs_augru_fwd / rs_augru_bwd against `augru` below, a float64 restatement (the reference has no AUGRU): h_all,
    d_gi, d_gh, d_att; att == 1 is the GRU, att == 0 keeps h at exactly zero; the inference forward equals the training
    forward; d_att is reproducible.
  * RS_DIN_WEIGHTS on both kernel families: the output is bit for bit the attw of the other modes, the backward matches
    the float64 softmax weights of oracle.interactions.din_attention, tensor cores agree with CUDA cores.
  * model.DIEN(evolution="augru") against a float64 autograd restatement, fused rows, determinism, the default mode.
  * The C4 shape (1 M items, B = 8192, L = 100, D = 64, fused rows, SGD) against the float64 step reference of
    test_c3_c4_shapes_gpu with the kernels' ReLU masks, and graph replay against eager.
The float64 restatements and the option checks run without a GPU.
"""
import gc
import os

import numpy as np
import pytest
import torch

from oracle import interactions as OI
from test_c3_c4_shapes_gpu import (C4_B, C4_D, C4_GB, C4_ITEMS, C4_L, C4_LR, _dense_params, _din_unit, _fc, c4_batch, reference,
                                   run_steps)
from test_full_scale_gpu import big_case, need_free  # noqa: F401

gpu = pytest.mark.gpu


def close(got, want, rtol=1e-5, atol=1e-6, msg=""):
    np.testing.assert_allclose(got.detach().cpu().double().numpy(), want.detach().cpu().double().numpy(), rtol=rtol, atol=atol,
                               err_msg=msg)


def _gru_weights(g, D, H, dtype=torch.float64):
    k = 1.0 / H ** 0.5
    w_ih, w_hh = [(torch.rand(3 * H, n, generator=g, dtype=dtype) * 2 - 1) * k for n in (D, H)]
    b_ih, b_hh = [(torch.rand(3 * H, generator=g, dtype=dtype) * 2 - 1) * k for _ in range(2)]
    return w_ih, w_hh, b_ih, b_hh


def augru(x, att, w_ih, w_hh, b_ih, b_hh):
    """The DIEN paper's attention-gated GRU in torch's gate convention, h0 = 0, next to oracle.interactions.gru:
    u = att[:, s] (1 - z),  h = (1 - u) h + u n.  x (B, L, D) unscaled, att (B, L) -> final hidden (B, H), in x's dtype
    and on x's device."""
    B, L, _ = x.shape
    H = w_hh.shape[1]
    h = x.new_zeros(B, H)
    for s in range(L):
        gi = x[:, s] @ w_ih.t() + b_ih
        gh = h @ w_hh.t() + b_hh
        ir, iz, inn = gi.split(H, dim=1)
        hr, hz, hn = gh.split(H, dim=1)
        r = torch.sigmoid(ir + hr)
        z = torch.sigmoid(iz + hz)
        n = torch.tanh(inn + r * hn)
        u = att[:, s:s + 1] * (1.0 - z)
        h = (1.0 - u) * h + u * n
    return h


def _augru_all(gi, att, w_hh, b_hh):
    """every h_t of the AUGRU on input projections gi (B, L, 3H): augru's loop, kept per step"""
    B, L, H3 = gi.shape
    H = H3 // 3
    h, hs = gi.new_zeros(B, H), []
    for s in range(L):
        gh = h @ w_hh.t() + b_hh
        ir, iz, inn = gi[:, s].split(H, dim=1)
        hr, hz, hn = gh.split(H, dim=1)
        r, z = torch.sigmoid(ir + hr), torch.sigmoid(iz + hz)
        n = torch.tanh(inn + r * hn)
        u = att[:, s:s + 1] * (1.0 - z)
        h = (1.0 - u) * h + u * n
        hs.append(h)
    return torch.stack(hs, dim=1)


# ---------------------------------------------------------------------------------------------- CPU: the restatements
def test_augru_oracle_limits():
    """augru: att == 1 is oracle.interactions.gru (and so nn.GRU), att == 0 gives exactly zero"""
    g = torch.Generator().manual_seed(1)
    B, L, D, H = 9, 6, 5, 8
    x = torch.randn(B, L, D, generator=g, dtype=torch.float64)
    ws = _gru_weights(g, D, H)
    torch.testing.assert_close(augru(x, torch.ones(B, L, dtype=torch.float64), *ws), OI.gru(x, *ws), rtol=1e-14, atol=1e-15)
    assert not bool(augru(x, torch.zeros(B, L, dtype=torch.float64), *ws).any())
    att = torch.rand(B, L, generator=g, dtype=torch.float64)
    gi = x @ ws[0].t() + ws[2]
    assert torch.equal(_augru_all(gi, att, ws[1], ws[3])[:, -1], augru(x, att, *ws))


def test_dien_evolution_option():
    from deeplearningrecommendationsystem_b200 import model as M
    with pytest.raises(ValueError):
        M.DIEN(10, 16, evolution="agru")
    torch.manual_seed(0)
    a = M.DIEN(10, 16)
    torch.manual_seed(0)
    b = M.DIEN(10, 16, evolution="augru")
    sa, sb = a.state_dict(), b.state_dict()
    assert list(sa) == list(sb) and all(sa[k].shape == sb[k].shape and torch.equal(sa[k], sb[k]) for k in sa)
    assert a.evolution == "gru"


def dien_augru_logit(P, X, M, am, tr):
    """model.DIEN(evolution="augru"): softmax weights w of the attention unit gate the GRU's update over the unscaled
    history, u = w_t (1 - z), h = (1 - u) h + u n; fc on [h_L, target].  In the mass pass the gates and weights keep
    their real values and pass on the magnitude of their derivative (|d u / d z| = w, |d h / d u| <= |n| + |h|)."""
    checks = []
    L = X.shape[1] - 1
    w = _din_unit(P, X, M, am, tr, "din.", checks)
    gi = X[:, :L] @ P["interest_evolution.weight_ih_l0"].t() + P["interest_evolution.bias_ih_l0"]
    Whh, bhh = P["interest_evolution.weight_hh_l0"], P["interest_evolution.bias_hh_l0"]
    H = Whh.shape[1]
    hs = X.new_zeros(X.shape[0], H)
    for s in range(L):
        gh = hs @ Whh.t() + bhh
        xr, xz = gi[:, s, :H] + gh[:, :H], gi[:, s, H:2 * H] + gh[:, H:2 * H]
        a = w[:, s:s + 1]
        if not am:
            r, z = torch.sigmoid(xr), torch.sigmoid(xz)
            n = torch.tanh(gi[:, s, 2 * H:] + r * gh[:, 2 * H:])
            tr[s] = (r.detach(), z.detach(), n.detach())
            u = a * (1.0 - z)
            hs = (1.0 - u) * hs + u * n
        else:
            r0, z0, n0 = tr[s]
            r = r0 + r0 * (1 - r0) * (xr - xr.detach())
            z = z0 + z0 * (1 - z0) * (xz - xz.detach())
            xn = gi[:, s, 2 * H:] + r * gh[:, 2 * H:]
            n = n0.abs() + (1 - n0 * n0) * (xn - xn.detach())
            a0 = a.detach()
            u0 = a0 * (1 - z0)
            du = (1 - z0) * (a - a0) + a0 * (z - z.detach())
            hs = (1.0 - u0) * hs + u0 * n + du * (n.detach() + hs.detach())
    return _fc(P, torch.cat([hs, X[:, L]], dim=1), M, am, checks), checks


def _dien64(sd, hist, tgt):
    """model.DIEN(evolution="augru") restated from its state dict with oracle.interactions and augru, in sd's dtype"""
    tab = sd["din.item_embedding.weight"]
    h, t = tab[hist], tab[tgt]
    att = OI.din_attention(h, t, [(sd[f"din.attention.{k}.weight"], sd[f"din.attention.{k}.bias"]) for k in (0, 2, 4)])
    hL = augru(h, att, sd["interest_evolution.weight_ih_l0"], sd["interest_evolution.weight_hh_l0"],
               sd["interest_evolution.bias_ih_l0"], sd["interest_evolution.bias_hh_l0"])
    f = OI.relu_tower(torch.cat([hL, t], dim=1), [(sd[f"fc.{k}.weight"], sd[f"fc.{k}.bias"]) for k in (0, 2, 4)], relu_last=False)
    return torch.sigmoid(f).view(-1)


def test_dien_augru_reference_matches_the_oracle():
    """the C4 step reference with dien_augru_logit and masks = (z > 0), float64 on the CPU, against autograd of the
    restatement from oracle.interactions and augru: predictions, loss, every dense gradient and the summed row
    gradient to 1e-12; the mass pass bounds every gradient"""
    from deeplearningrecommendationsystem_b200 import model as M
    torch.manual_seed(3)
    items, D, L, nb = 60, 8, 7, 200
    m = M.DIEN(items, D, evolution="augru").double()
    with torch.no_grad():
        for n, p in m.named_parameters():
            if n.endswith("bias"):
                p.normal_(0.0, 0.2)
    sd = {k: v.detach().clone() for k, v in m.state_dict().items()}
    g = torch.Generator().manual_seed(9)
    hist, tgt = torch.randint(0, items, (nb, L), generator=g), torch.randint(0, items, (nb,), generator=g)
    y = (torch.rand(nb, generator=g) < 0.4).double()
    tab = sd["din.item_embedding.weight"]
    h, t = tab[hist], tab[tgt]
    x = torch.cat([h, h - t.unsqueeze(1), t.unsqueeze(1).expand_as(h)], dim=-1)
    z0 = x @ sd["din.attention.0.weight"].t() + sd["din.attention.0.bias"]
    z1 = torch.relu(z0) @ sd["din.attention.2.weight"].t() + sd["din.attention.2.bias"]
    w = torch.softmax((torch.relu(z1) @ sd["din.attention.4.weight"].t() + sd["din.attention.4.bias"]).squeeze(-1), dim=-1)
    ev = m.interest_evolution
    hL = augru(h, w, ev.weight_ih_l0.detach(), ev.weight_hh_l0.detach(), ev.bias_ih_l0.detach(), ev.bias_hh_l0.detach())
    a = torch.cat([hL, t], dim=1) @ sd["fc.0.weight"].t() + sd["fc.0.bias"]
    b = torch.relu(a) @ sd["fc.2.weight"].t() + sd["fc.2.bias"]
    masks = {"act0": z0 > 0, "act1": z1 > 0, "act0_val": torch.relu(z0), "act1_val": torch.relu(z1), "attw_val": w, "fc.1": a > 0,
             "fc.3": b > 0}
    leaves = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    pred = _dien64(leaves, hist, tgt)
    loss = OI.bce(pred, y)
    params = {k: v for k, v in sd.items() if not k.endswith("item_embedding.weight")}
    got = torch.autograd.grad(loss, [leaves["din.item_embedding.weight"]] + [leaves[k] for k in params])
    keys = torch.cat([hist, tgt.unsqueeze(1)], dim=1)
    uniq, inv = torch.unique(keys, return_inverse=True)
    ref = reference(dien_augru_logit, params, tab[uniq], inv, y, masks, chunk=70)
    c = lambda a, b, what: np.testing.assert_allclose(a.detach().numpy(), b.detach().numpy(), rtol=1e-12, atol=1e-15, err_msg=what)  # noqa: E731
    c(ref["pred"], pred, "pred")
    c(ref["loss"], loss, "loss")
    c(ref["g_rows"], got[0][uniq], "rows")
    for k, gk in zip(params, got[1:]):
        c(ref["grads"][k], gk, k)
        assert bool((ref["mass"][k] >= gk.abs() * (1 - 1e-12)).all()), k
    assert bool((ref["S"] >= ref["S_plain"] * (1 - 1e-12)).all()) and bool((ref["S_plain"] >= ref["g_rows"].abs() * (1 - 1e-12)).all())


# ---------------------------------------------------------------------------------------------- kernels
@gpu
@pytest.mark.parametrize("L", [1, 3, 100])
@pytest.mark.parametrize("H,B", [(8, 17), (16, 50), (32, 33), (64, 21)])
def test_augru_kernels_match_float64(H, B, L):
    from deeplearningrecommendationsystem_b200 import ops
    g = torch.Generator().manual_seed(7 * H + L)
    ws = _gru_weights(g, 3 * H, H)
    _, w_hh, _, b_hh = ws
    gi = (torch.randn(B, L, 3 * H, generator=g, dtype=torch.float64) * 0.7).requires_grad_(True)
    att = torch.rand(B, L, generator=g, dtype=torch.float64).requires_grad_(True)
    w_hh, b_hh = w_hh.requires_grad_(True), b_hh.requires_grad_(True)
    want = _augru_all(gi, att, w_hh, b_hh)
    eye = torch.eye(3 * H, dtype=torch.float64)           # the oracle with W_ih = I, b_ih = 0 takes gi as its input
    assert torch.equal(want[:, -1], augru(gi, att, eye, w_hh, torch.zeros(3 * H, dtype=torch.float64), b_hh))
    g_all, g_last = torch.randn(B, L, H, generator=g, dtype=torch.float64), torch.randn(B, H, generator=g, dtype=torch.float64)
    grads = torch.autograd.grad((want * g_all).sum() + (want[:, -1] * g_last).sum(), [gi, att, w_hh, b_hh])
    c32 = lambda t: t.detach().float().cuda()              # noqa: E731
    h_all, gates = ops.augru_fwd(c32(gi), c32(att), c32(w_hh), c32(b_hh))
    close(h_all, want, msg="h_all")
    h_inf, none = ops.augru_fwd(c32(gi), c32(att), c32(w_hh), c32(b_hh), want_gates=False)
    assert none is None and torch.equal(h_inf, h_all), "inference forward differs from the training forward"
    d_gi, d_gh, d_att = ops.augru_bwd(c32(w_hh), c32(att), h_all, gates, g_h_all=c32(g_all), g_h_last=c32(g_last))
    h_prev = torch.cat([torch.zeros(B, 1, H), h_all.cpu()[:, :-1]], dim=1).double()
    d_gh64 = d_gh.cpu().double().reshape(-1, 3 * H)
    got = {"d_gi": d_gi, "d_att": d_att, "dW_hh (d_gh)": d_gh64.t() @ h_prev.reshape(-1, H), "db_hh (d_gh)": d_gh64.sum(0)}
    for (name, a), w_ in zip(got.items(), grads):
        close(a, w_, rtol=1e-5, atol=2e-6 * max(1.0, float(w_.abs().max())), msg=name)
    # d_gh: the r and z columns are those of d_gi; the n columns are d gi_n * r
    r = gates.view(B, L, 4, H)[:, :, 0]
    assert torch.equal(d_gh[..., :2 * H], d_gi[..., :2 * H])
    assert torch.equal(d_gh[..., 2 * H:], d_gi[..., 2 * H:] * r)
    again = ops.augru_bwd(c32(w_hh), c32(att), h_all, gates, g_h_all=c32(g_all), g_h_last=c32(g_last))
    assert all(torch.equal(a, b) for a, b in zip((d_gi, d_gh, d_att), again)), "the backward is not reproducible"


@gpu
@pytest.mark.parametrize("H,B,L", [(8, 17, 3), (64, 21, 100), (32, 33, 1)])
def test_augru_limits_equal_the_gru(H, B, L):
    """att == 1: rs_augru_* equal rs_gru_* and nn.GRU to 1e-5; att == 0: h_all is exactly zero"""
    from deeplearningrecommendationsystem_b200 import ops
    g = torch.Generator().manual_seed(H + B)
    x = torch.randn(B, L, H, generator=g) * 0.5
    ref = torch.nn.GRU(H, H, batch_first=True)
    gi = torch.nn.functional.linear(x, ref.weight_ih_l0, ref.bias_ih_l0).detach().cuda()
    w_hh, b_hh = ref.weight_hh_l0.detach().cuda(), ref.bias_hh_l0.detach().cuda()
    gl = torch.randn(B, H, generator=g).cuda()
    h_gru, gates_gru = ops.gru_fwd(gi, w_hh, b_hh)
    h_au, gates_au = ops.augru_fwd(gi, torch.ones(B, L, device="cuda"), w_hh, b_hh)
    close(h_au, h_gru, msg="h_all vs rs_gru_fwd")
    with torch.no_grad():
        close(h_au[:, -1], ref(x)[1][-1], msg="h_L vs nn.GRU")
    d_gi, d_gh = ops.gru_bwd(w_hh, h_gru, gates_gru, g_h_last=gl)
    a_gi, a_gh, _ = ops.augru_bwd(w_hh, torch.ones(B, L, device="cuda"), h_au, gates_au, g_h_last=gl)
    close(a_gi, d_gi, atol=1e-6 * max(1.0, float(d_gi.abs().max())), msg="d_gi vs rs_gru_bwd")
    close(a_gh, d_gh, atol=1e-6 * max(1.0, float(d_gh.abs().max())), msg="d_gh vs rs_gru_bwd")
    h0, _ = ops.augru_fwd(gi, torch.zeros(B, L, device="cuda"), w_hh, b_hh)
    assert not bool(h0.any()), "att == 0 must keep every h_t at zero"


@gpu
def test_augru_rejects_bad_shapes():
    from deeplearningrecommendationsystem_b200 import attention, ops
    gru = torch.nn.GRU(16, 16, batch_first=True).cuda()
    x = torch.randn(4, 5, 16, device="cuda")
    with pytest.raises(ValueError):
        attention.augru_last_hidden(x, torch.rand(4, 6, device="cuda"), gru)
    with pytest.raises(NotImplementedError):
        attention.augru_last_hidden(torch.randn(4, 5, 12, device="cuda"), torch.rand(4, 5, device="cuda"),
                                    torch.nn.GRU(12, 12, batch_first=True).cuda())
    with pytest.raises(RuntimeError):                      # the CTA's attention block does not fit shared memory
        ops.augru_fwd(torch.zeros(1, 4000, 192, device="cuda"), torch.zeros(1, 4000, device="cuda"), gru.weight_hh_l0.detach(),
                      gru.bias_hh_l0.detach())


# ---------------------------------------------------------------------------------------------- the weights mode
def _din_case(g, B, L, D, H1=64, H2=32):
    rows = torch.randn(B, L + 1, D, generator=g, dtype=torch.float64) * 0.5
    lin = lambda o, i: (torch.rand(o, i, generator=g, dtype=torch.float64) * 2 - 1) / i ** 0.5   # noqa: E731
    vec = lambda o, i: (torch.rand(o, generator=g, dtype=torch.float64) * 2 - 1) / i ** 0.5      # noqa: E731
    return rows, [lin(H1, 3 * D), vec(H1, 3 * D), lin(H2, H1), vec(H2, H1), lin(1, H2), vec(1, H2)]


def _weights64(rows, ws, masks=None):
    """oracle.interactions.din_attention, or (masks = (m0, m1)) the same unit with every ReLU z * mask; also returns the
    pre-activations (z0, z1)"""
    h, t = rows[:, :-1], rows[:, -1]
    te = t.unsqueeze(1).expand_as(h)
    z0 = torch.cat([h, h - te, te], dim=-1) @ ws[0].t() + ws[1]
    a0 = torch.relu(z0) if masks is None else z0 * masks[0]
    z1 = a0 @ ws[2].t() + ws[3]
    a1 = torch.relu(z1) if masks is None else z1 * masks[1]
    return torch.softmax((a1 @ ws[4].t() + ws[5]).squeeze(-1), dim=-1), (z0, z1)


@gpu
@pytest.mark.parametrize("impl", ["fused", "tc"])
@pytest.mark.parametrize("D,H1,H2,L,B", [(16, 64, 32, 7, 90), (64, 64, 32, 100, 20), (32, 128, 64, 33, 40), (64, 128, 64, 100, 300)])
def test_din_weights_mode_matches_float64(impl, D, H1, H2, L, B):
    from deeplearningrecommendationsystem_b200 import ops
    g = torch.Generator().manual_seed(D + L + H1)
    rows, ws = _din_case(g, B, L, D, H1, H2)
    rows, ws = rows.requires_grad_(True), [w.requires_grad_(True) for w in ws]
    w = OI.din_attention(rows[:, :-1], rows[:, -1], [(ws[0], ws[1]), (ws[2], ws[3]), (ws[4], ws[5])])
    gup = torch.randn(B, L, generator=g, dtype=torch.float64)
    r32, cw = rows.detach().float().cuda(), [t.detach().float().cuda() for t in ws]
    out, attw, stash = ops.din_fwd(r32, cw, ops.DIN_WEIGHTS, want_attw=True, impl=impl, want_stash=True)
    assert out.shape == (B, L) and attw is out
    assert (stash is not None) == (impl == "tc")
    if impl == "tc":
        # ReLU is not differentiable at 0: over B L = 30 000 rows a pre-activation within rounding of zero may land on the
        # other side in 3xTF32 than in float64, which moves that (b, l) row's gradient by a finite amount.  So the masks
        # the forward stashed may differ from float64's only there, and the backward is checked with those masks fixed.
        masks = tuple((a.view(B, L, -1) > 0).cpu().double() for a in stash[1:])
        w_fixed, zs = _weights64(rows, ws, masks)
        for m, z in zip(masks, zs):
            flip = m != (z.detach() > 0).double()
            assert int(flip.any(-1).sum()) <= max(2, int(2e-4 * B * L)), "stashed ReLU masks differ from float64"
            if bool(flip.any()):
                assert float(z.detach()[flip].abs().max()) <= 1e-5 * float(z.detach().abs().max()), "a flipped mask bit away from 0"
        grads = torch.autograd.grad((w_fixed * gup).sum(), [rows] + ws)
    else:
        grads = torch.autograd.grad((w * gup).sum(), [rows] + ws)
    for pool in (True, False):
        _, attw_other = ops.din_fwd(r32, cw, pool, want_attw=True, impl=impl)
        assert torch.equal(out, attw_other), f"weights differ from the attw of pool={pool}"
    out2, none = ops.din_fwd(r32, cw, ops.DIN_WEIGHTS, impl=impl)
    assert none is None and torch.equal(out2, out)

    def scaled(got, ref, name):
        close(got, ref, rtol=1e-5, atol=1e-5 * max(1e-3, float(ref.abs().max())), msg=f"{name} ({impl})")
    scaled(out, w.detach(), "w")
    if impl == "tc":
        d_rows, dws = ops.din_bwd_tc(r32, cw, ops.DIN_WEIGHTS, gup.float().cuda(), stash)
    else:
        d_rows, dws = ops.din_bwd(r32, cw, ops.DIN_WEIGHTS, gup.float().cuda())
    scaled(d_rows, grads[0], "d_rows")
    for got, ref, name in zip(dws[:5], grads[1:6], ["dW0", "db0", "dW1", "db1", "dW2"]):
        assert got.shape == ref.shape, name
        scaled(got, ref, name)
    assert float(dws[5].abs().max()) <= 1e-5 * max(1e-3, float(grads[5].abs().max()), float(grads[4].abs().max()))


@gpu
def test_din_weights_tc_equals_fused():
    """din_attention_weights through autograd: the tcgen05 kernels and the CUDA-core pair (RS_DIN_TC=0) agree"""
    from deeplearningrecommendationsystem_b200 import attention, ops
    g = torch.Generator().manual_seed(0)
    B, L, D = 90, 100, 64
    unit = torch.nn.Sequential(torch.nn.Linear(3 * D, 64), torch.nn.ReLU(), torch.nn.Linear(64, 32), torch.nn.ReLU(),
                               torch.nn.Linear(32, 1)).cuda()
    rows = (torch.randn(B, L + 1, D, generator=g) * 0.5).cuda()
    gup = torch.randn(B, L, generator=g).cuda()
    res = {}
    for impl in ("tc", "fused"):
        if impl == "fused":
            os.environ["RS_DIN_TC"] = "0"
        try:
            r = rows.clone().requires_grad_(True)
            unit.zero_grad()
            n0 = ops.launches()
            out = attention.din_attention_weights(r, unit)
            (out * gup).sum().backward()
            res[impl] = [out.detach(), r.grad] + [p.grad.clone() for p in unit.parameters()]
            res[impl + "_launches"] = ops.launches() - n0
        finally:
            os.environ.pop("RS_DIN_TC", None)
    assert res["tc_launches"] > res["fused_launches"]
    for k, (a, b) in enumerate(list(zip(res["tc"], res["fused"]))[:-1]):
        tol = 1e-5 * max(1e-3, float(b.abs().max()))
        if k == 1:
            bad = int(((a - b).abs() > tol + 1e-5 * b.abs()).flatten(1).any(dim=1).sum())
            assert bad <= 1, f"{bad} samples differ"
        else:
            assert float((a - b).norm()) <= 1e-4 * float(b.norm()) + tol, k


# ---------------------------------------------------------------------------------------------- the model
SMALL = dict(items=300, D=16, L=7, B=200)


def _small_model(evolution="augru", seed=0):
    from deeplearningrecommendationsystem_b200 import model as M
    torch.manual_seed(seed)
    m = M.DIEN(SMALL["items"], SMALL["D"], evolution=evolution)
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


@gpu
def test_small_dien_augru_matches_float64():
    """predictions, loss and every gradient against autograd of the float64 restatement; then two torch-Adam steps"""
    m = _small_model()
    sd64 = {k: v.detach().double().clone().requires_grad_(True) for k, v in m.state_dict().items()}
    m = m.cuda()
    hist, tgt, y = _small_batch(1)
    lr = 1e-3
    opt = torch.optim.Adam(m.parameters(), lr=lr)
    opt64 = torch.optim.Adam(list(sd64.values()), lr=lr)
    names = [n for n, _ in m.named_parameters()]
    first = None
    for step in range(2):
        opt.zero_grad()
        opt64.zero_grad()
        p = m(hist.cuda(), tgt.cuda())
        loss = torch.nn.BCELoss()(p, y.cuda())
        loss.backward()
        p64 = _dien64(sd64, hist, tgt)
        loss64 = OI.bce(p64, y.view(-1).double())
        loss64.backward()
        close(p.view(-1), p64, msg=f"step {step} pred")
        close(loss, loss64, msg=f"step {step} loss")
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
    # Adam moves every element by about lr whatever the gradient's size, so an element whose gradient is within rounding
    # of zero may move either way; the others must agree closely
    for n, q in m.named_parameters():
        settled = first[n] > 1e-2 * float(first[n].max())
        err = (q.detach().cpu().double() - sd64[n].detach()).abs()
        if bool(settled.any()):
            assert float(err[settled].max()) <= 1e-3 * lr + 1e-6 * float(sd64[n].detach().abs().max()), n
        assert float(err.max()) <= 4 * lr, n


@gpu
def test_small_dien_augru_fused_rows_and_determinism():
    """fused sparse rows with SGD give the parameters of SGD on dense tables; the table gradient is bitwise
    deterministic; evolution="gru" is bit-identical to the default; recommendation() ranks the model's own scores"""
    from deeplearningrecommendationsystem_b200.optim import FusedRowOptimizer
    from deeplearningrecommendationsystem_b200.trainer import Trainer
    lr = 0.05
    dense, fused = _small_model().cuda(), _small_model().cuda().fuse_embedding_updates()
    tr_d = Trainer(dense, torch.nn.BCELoss(), torch.optim.SGD(dense.parameters(), lr=lr))
    tr_f = Trainer(fused, torch.nn.BCELoss(), FusedRowOptimizer(fused, torch.optim.SGD(
        [p for p in fused.parameters() if p.requires_grad], lr=lr), lr=lr, kind="sgd"))
    for step in range(2):
        hist, tgt, y = _small_batch(10 + step)
        tr_d.train_loop(hist.cuda(), tgt.cuda(), train_rating=y.cuda())
        tr_f.train_loop(hist.cuda(), tgt.cuda(), train_rating=y.cuda())
        close(tr_f.predictions_train, tr_d.predictions_train, msg=f"step {step} pred")
    for (n, a), (_, b) in zip(dense.state_dict().items(), fused.state_dict().items()):
        close(b, a, rtol=1e-5, atol=1e-6, msg=n)
    hist, tgt, y = (t.cuda() for t in _small_batch(20))
    gs = []
    for _ in range(2):
        dense.zero_grad()
        torch.nn.BCELoss()(dense(hist, tgt), y).backward()
        gs.append(dense.din.item_embedding.weight.grad.clone())
    assert torch.equal(gs[0], gs[1]), "the table gradient is not deterministic"
    from deeplearningrecommendationsystem_b200 import model as M
    from deeplearningrecommendationsystem_b200.model import _blocks as K
    outs = []
    for kw in ({}, {"evolution": "gru"}):
        torch.manual_seed(5)
        m = M.DIEN(SMALL["items"], SMALL["D"], **kw).cuda()
        p = m(hist, tgt)
        torch.nn.BCELoss()(p, y).backward()
        outs.append([p.detach()] + [q.grad.clone() for q in m.parameters()])
    assert all(torch.equal(u, v) for u, v in zip(*outs)), "evolution='gru' differs from the default"
    # recommendation(): the catalogue is scored in one chunk here, so the same forward gives the same scores
    m = _small_model().cuda().eval()
    hist_list = _small_batch(30)[0][:6].tolist()
    k = 10
    got = m.recommendation(6, SMALL["items"], hist_list, k)
    assert got.shape == (6, k)
    with torch.no_grad():
        s = K.history_scores(m, hist_list, SMALL["items"], torch.device("cuda"))(0, 6).view(6, SMALL["items"])
    for u in range(6):
        assert torch.equal(s[u][torch.as_tensor(got[u], device="cuda")], torch.topk(s[u], k).values), f"user {u}"


# ---------------------------------------------------------------------------------------------- the C4 shape
def _c4_augru(seed=0):
    from deeplearningrecommendationsystem_b200 import model as M
    from deeplearningrecommendationsystem_b200.optim import FusedRowOptimizer
    torch.manual_seed(seed)
    m = M.DIEN(C4_ITEMS, C4_D, evolution="augru").cuda().fuse_embedding_updates()
    return m, FusedRowOptimizer(m, torch.optim.SGD([p for p in m.parameters() if p.requires_grad], lr=C4_LR), lr=C4_LR, kind="sgd")


@gpu
def test_c4_augru_step_matches_float64(big_case, monkeypatch):
    """DIEN(1 M items, 64, evolution="augru") at B = 8192, L = 100, lr 0.01, fused rows + SGD: two steps of
    Trainer.train_loop against the float64 reference with the kernels' ReLU masks; untouched rows stay bit-identical"""
    from deeplearningrecommendationsystem_b200 import ops
    from deeplearningrecommendationsystem_b200.trainer import Trainer
    free = need_free(C4_GB)
    ins, y = c4_batch(53)
    m, opt = _c4_augru()
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
    keys = torch.cat([ins[0], ins[1].unsqueeze(1)], dim=1)
    info = run_steps("c4 dien augru", m, tr, ins, y, m.din.item_embedding.weight.data, keys, _dense_params(m), dien_augru_logit,
                     capture, 2048, C4_LR)
    big_case["info"] = f"c4 dien augru: {free}, {info}"


@gpu
def test_c4_augru_graphed_step_equals_eager(big_case):
    from deeplearningrecommendationsystem_b200.graph import GraphedTrainStep
    from deeplearningrecommendationsystem_b200.trainer import Trainer
    free = need_free(C4_GB)
    (m1, o1), (m2, o2) = _c4_augru(4), _c4_augru(4)
    big_case["model"] = (m1, m2)
    tr = Trainer(m1, torch.nn.BCELoss(), o1)
    gs = GraphedTrainStep(m2, torch.nn.BCELoss(), o2, warmup=1)
    for k in range(3):
        ins, y = c4_batch(80 + k)
        tr.train_loop(*ins, train_rating=y)
        pred, loss = gs(*ins, rating=y)
        assert torch.equal(pred, tr.predictions_train), f"step {k}: predictions differ"
        assert torch.equal(loss, tr.train_loss), f"step {k}: losses differ"
    assert gs.graph is not None
    for (n, a), (_, b) in zip(m1.named_parameters(), m2.named_parameters()):
        assert torch.equal(a, b), f"{n} differs between the graphed and the eager step"
    assert torch.equal(m1.din.item_embedding.weight, m2.din.item_embedding.weight)
    big_case["info"] = f"graphed == eager dien augru: {free}"
    del gs, tr
    gc.collect()
