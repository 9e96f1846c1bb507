"""The C3 (PNN / AFM over 39 Criteo-shaped fields, D = 32, B = 32768) and C4 (DIN / DIEN, 1 M-row item table, L = 100,
D = 64, B = 8192) train steps at the shapes bench.py times, each checked against a float64 reference of the same step.

Every other test of afm_tc.cu, din_tc.cu and gru.cu runs far below these sizes, so their persistent loops turn a few
times at most: here the AFM kernels take ~74-111 samples per warpgroup (afm_de_kernel: ~5.5 per warp, so its
grid-stride loop steps), the DIN tensor-core kernels ~22 128-row tiles per warpgroup and the GRU kernels 512 CTAs.

These steps have ReLUs everywhere (AFM attention, DIN / DIEN attention units, PNN / DIN / DIEN towers), and with
1.55e9 AFM pre-activations per batch some sit within rounding of zero: a float64 reference that took its own ReLU
decisions would disagree with any correct fp32 kernel by a finite amount.  So the reference (`reference`) uses the
kernels' own masks -- every ReLU is z * mask -- and with fixed masks the gradient is a smooth function of the inputs,
which allows an element-wise bar everywhere.  The masks are borrowed without changing the library:
  * AFM attention: ops.afm_bwd is wrapped to run with return_masks=True (the bits its chain kernel used);
  * DIN / DIEN attention unit: ops.din_fwd is wrapped to keep the stash (attw, act0, act1); masks act0 > 0, act1 > 0
    are what din_bwd_tc consumes;
  * torch towers: forward hooks (FieldPNN.dnn_network[k]: pre-activation z, mask z > 0 = torch.relu's backward mask;
    DIN / DIEN fc ReLU modules: output, mask out > 0).
Borrowed masks must not hide a mask bug: every mask must equal (z64 > 0) wherever |z64| exceeds 1e-5 of the |.|-mass of
that pre-activation (|x| |W|^T + |b|), the entries inside that band must be a small fraction, and the DIN stash
itself (act0, act1, attw) must match its float64 values.

Bounds.  Rows: assert_rows_match of test_full_scale_gpu, |w - w64| <= 1e-6 |w64| + lr (1e-5 |g64| + 4 eps32 S), where
S sums the |.|-mass of each lookup's gradient term.  The term a kernel hands to the row update is itself an fp32 sum
with possible cancellation inside it (AFM: 38 partners x (a 64-term dz W^T + w g); PNN: 38 pair terms plus a 256-term
column of dh0 W1; DIN: a 128-term dz0 W0 behind the softmax backward; DIEN: the same, behind a 100-step BPTT), so its
rounding is relative to the magnitude of its constituents, not to its value.  That mass is what `reference` computes
in its second pass: the same step with every weight, input and upstream gradient replaced by its magnitude and every
nonlinearity by the magnitude of its derivative at the real point (softmax: w (x + sum w x) instead of
w (x - sum w x)), i.e. the constituent mass of each gradient, propagated through the whole chain.  Dense parameters:
|grad - g64| <= 1e-5 |g64| + 8 eps32 M with M that mass; 8 rather than 4 because the AFM and DIN weight gradients are
3xTF32 tensor-core products, each carrying up to ~12 eps32 of relative error (uncorrelated, so a few eps32 of the
mass over a sum).  The AFM attention parameters are the exception, see afm_dw_floor.  The report gives the worst error / bound per group, and for the rows also against the plain
bound (S = sum of |term|), which shows whether the mass was needed.
"""
import gc

import numpy as np
import pytest
import torch

from test_full_scale_gpu import C2_CARDS, EPS32, assert_rows_match, big_case, guard_rows, make_batch, need_free, zipf_ids  # noqa: F401

C3_CARDS = C2_CARDS + [64] * 13
C3_B, C3_D, C3_LR = 32768, 32, 0.05
C4_ITEMS, C4_B, C4_L, C4_D, C4_LR = 1_000_000, 8192, 100, 64, 0.01
DENSE_EPS = 8               # dense-gradient floor: DENSE_EPS eps32 of the constituent mass (see the module docstring)
BAND = 1e-5                 # |z64| <= BAND x mass(z): a ReLU decision fp32 may take either way
BAND_FRACTION = 1e-3        # ... and at most this fraction of the pre-activations of one kind may sit there
C3_GB, C4_GB = 40, 30       # device memory a case needs, with margin (table(s), AFM workspace + masks, reference chunk)


# ---------------------------------------------------------------------------------------------- the float64 reference
def _lin(x, P, name):
    return x @ P[name + ".weight"].t() + P[name + ".bias"]


def _lin_mass(x, P, name):
    return x.detach().abs() @ P[name + ".weight"].detach().abs().t() + P[name + ".bias"].detach().abs()


def _softmax(s, am, tr, key):
    """softmax over the last dim; in the mass pass a stand-in with the real weights w as value and Jacobian
    diag(w) + w w^T (the magnitude of softmax's diag(w) - w w^T): upstream x -> w (x + sum w x)"""
    if not am:
        w = torch.softmax(s, dim=-1)
        tr[key] = w.detach()
        return w
    w = tr[key]
    d = s - s.detach()
    return w * (1.0 + d) + w * (w * d).sum(-1, keepdim=True)


def _pairs(F, device):
    iu = torch.triu_indices(F, F, offset=1, device=device)
    return iu[0], iu[1]


def pnn_logit(P, X, M, am, tr):
    """FieldPNN: X (c, F, D) rows of the lookups; M: the dnn_network masks"""
    c, F, D = X.shape
    i, j = _pairs(F, X.device)
    h = _lin(X.reshape(c, F * D), P, "linear1") + _lin((X[:, i] * X[:, j]).sum(2), P, "linear2")
    checks, k = [], 0
    while f"dnn_network.{k}.weight" in P:
        name = f"dnn_network.{k}"
        z = _lin(h, P, name)
        if not am:
            checks.append((name, z.detach(), _lin_mass(h, P, name), M[name], None))
        h = z * M[name]
        k += 1
    return _lin(h, P, "output").view(-1), checks


def afm_logit(P, X, M, am, tr):
    """FieldAFM: X (c, F, D); M["attention"] (c, P, A): the ReLU bits of the tensor-core backward's chain kernel"""
    i, j = _pairs(X.shape[1], X.device)
    Pp = X[:, i] * X[:, j]                                            # (c, P, D)
    z = Pp @ P["attention_W"] + P["attention_b"]                      # (c, P, A)
    checks = []
    if not am:
        mass = Pp.detach().abs() @ P["attention_W"].detach().abs() + P["attention_b"].detach().abs()
        checks.append(("attention", z.detach(), mass, M["attention"], None))
    s = ((z * M["attention"]) @ P["attention_h"]).squeeze(-1)          # (c, P)
    w = _softmax(s, am, tr, "w")
    pooled = (w.unsqueeze(-1) * Pp).sum(1)
    return _lin(pooled, P, "output_layer").view(-1), checks


def _din_unit(P, X, M, am, tr, pfx, checks):
    """attention unit over [h, h - t, t] with the stashed masks -> softmax weights (c, L).  (The kernels evaluate the
    first layer concat-free, (Wa + Wb) h + (Wc - Wb) t; the concat form's mass is the larger of the two.)"""
    L = X.shape[1] - 1
    h, t = X[:, :L], X[:, L:].expand(-1, L, -1)
    x = torch.cat([h, h + t if am else h - t, t], dim=-1)
    z0 = _lin(x, P, pfx + "attention.0")
    z1 = _lin(z0 * M["act0"], P, pfx + "attention.2")
    if not am:
        checks.append(("attention.0", z0.detach(), _lin_mass(x, P, pfx + "attention.0"), M["act0"], M["act0_val"]))
        checks.append(("attention.2", z1.detach(), _lin_mass(z0 * M["act0"], P, pfx + "attention.2"), M["act1"], M["act1_val"]))
    s = _lin(z1 * M["act1"], P, pfx + "attention.4").squeeze(-1)
    w = _softmax(s, am, tr, "attw")
    if not am:
        checks.append(("attw", w.detach(), None, None, M["attw_val"]))
    return w


def _fc(P, f, M, am, checks):
    z = _lin(f, P, "fc.0")
    if not am:
        checks.append(("fc.0", z.detach(), _lin_mass(f, P, "fc.0"), M["fc.1"], None))
    a = z * M["fc.1"]
    z = _lin(a, P, "fc.2")
    if not am:
        checks.append(("fc.2", z.detach(), _lin_mass(a, P, "fc.2"), M["fc.3"], None))
    return _lin(z * M["fc.3"], P, "fc.4").view(-1)


def din_logit(P, X, M, am, tr):
    """model.DIN: X (c, L + 1, D) = [history | target] rows"""
    checks = []
    L = X.shape[1] - 1
    w = _din_unit(P, X, M, am, tr, "", checks)
    pooled = (X[:, :L] * w.unsqueeze(-1)).sum(1)
    return _fc(P, torch.cat([pooled, X[:, L]], dim=1), M, am, checks), checks


def dien_logit(P, X, M, am, tr):
    """model.DIEN: attention-scaled history -> nn.GRU (h0 = 0, gates r, z, n) -> fc on [h_L, target].  In the mass pass
    the gates keep their real values and pass on the magnitude of their derivative."""
    checks = []
    L = X.shape[1] - 1
    w = _din_unit(P, X, M, am, tr, "din.", checks)
    gi = (X[:, :L] * w.unsqueeze(-1)) @ P["interest_evolution.weight_ih_l0"].t() + P["interest_evolution.bias_ih_l0"]
    Whh, bhh = P["interest_evolution.weight_hh_l0"], P["interest_evolution.bias_hh_l0"]
    H = Whh.shape[1]
    hs = X.new_zeros(X.shape[0], H)
    for s in range(L):
        gh = hs @ Whh.t() + bhh
        xr, xz = gi[:, s, :H] + gh[:, :H], gi[:, s, H:2 * H] + gh[:, H:2 * H]
        if not am:
            r, z = torch.sigmoid(xr), torch.sigmoid(xz)
            n = torch.tanh(gi[:, s, 2 * H:] + r * gh[:, 2 * H:])
            tr[s] = (r.detach(), z.detach(), n.detach())
            hs = (1.0 - z) * n + z * hs
        else:
            r0, z0, n0 = tr[s]
            r = r0 + r0 * (1 - r0) * (xr - xr.detach())
            z = z0 + z0 * (1 - z0) * (xz - xz.detach())
            xn = gi[:, s, 2 * H:] + r * gh[:, 2 * H:]
            n = n0.abs() + (1 - n0 * n0) * (xn - xn.detach())
            hs = ((1.0 - z0) + (z - z.detach())) * n + z * hs
    return _fc(P, torch.cat([hs, X[:, L]], dim=1), M, am, checks), checks


def _check_masks(checks, stats):
    """mask == (z64 > 0) outside the near-zero band; stashed activations / weights within 1e-5 of float64"""
    for name, z, mass, mask, stash in checks:
        st = stats.setdefault(name, {"band": 0, "total": 0, "stash": 0.0})
        if mass is not None:
            band = z.abs() <= BAND * mass
            wrong = (mask != (z > 0)) & ~band
            if bool(wrong.any()):
                raise AssertionError(f"{name}: {int(wrong.sum())} ReLU mask bits disagree with float64 outside the near-zero band "
                                     f"(first |z|/mass {float((z.abs() / mass)[wrong][0]):.3e})")
            st["band"] += int(band.sum())
            st["total"] += z.numel()
        if stash is not None:
            want = z * mask if mask is not None else z
            err = (stash.double() - want).abs()
            bound = 1e-5 * want.abs() + 1e-5 * float(want.abs().max())
            assert bool((err <= bound).all()), f"{name}: stashed values off float64 by {float((err / bound).max()):.2f} of the bound"
            st["stash"] = max(st["stash"], float((err / bound).max()))


def reference(fwd, params, rows, inv, y, masks, chunk):
    """One step of a model in float64 (stock torch autograd, run where `rows` is), chunked over samples.

    fwd(P, X, M, am, tr) -> (logit (c,), checks): the model on the rows X (c, K, D) of a chunk's lookups with the masks
    M; am selects the mass pass (see the module docstring), tr carries the real pass's softmax weights and gates to it.
    params: the dense parameters before the step.  rows (U, D): the distinct table rows the batch looks up, before the
    step; inv (B, K): index into rows of each lookup.  masks: dict of (B, ...) tensors, sliced per chunk.
    Returns pred (B,), loss, grads / mass of every dense parameter, the summed row gradient g_rows (U, D), its
    constituent mass S (U, D), the plain sum of |per-lookup term| S_plain, and the mask statistics."""
    nb = inv.shape[0]
    P = {n: p.detach().double().requires_grad_(True) for n, p in params.items()}
    A = {n: p.detach().double().abs().requires_grad_(True) for n, p in params.items()}
    grads = {n: torch.zeros_like(p) for n, p in P.items()}
    mass = {n: torch.zeros_like(p) for n, p in P.items()}
    g_rows, S, S_plain = (torch.zeros(rows.shape, dtype=torch.float64, device=rows.device) for _ in range(3))
    pred = torch.empty(nb, dtype=torch.float64, device=rows.device)
    loss = torch.zeros((), dtype=torch.float64, device=rows.device)
    y64 = y.reshape(-1).double()
    stats = {}
    for s in range(0, nb, chunk):
        idx = inv[s:s + chunk]
        c = idx.shape[0]
        flat = idx.reshape(-1)
        M = {k: v[s:s + c] for k, v in masks.items()}
        tr = {}
        X = rows[idx].double().requires_grad_(True)
        logit, checks = fwd(P, X, M, False, tr)
        _check_masks(checks, stats)
        del checks
        p = torch.sigmoid(logit)
        yc = y64[s:s + c]
        lc = -(yc * torch.clamp(torch.log(p), min=-100.0) + (1.0 - yc) * torch.clamp(torch.log(1.0 - p), min=-100.0)).sum() / nb
        gs = torch.autograd.grad(lc, [X, *P.values()])
        g_rows.index_add_(0, flat, gs[0].reshape(flat.numel(), -1))
        S_plain.index_add_(0, flat, gs[0].abs().reshape(flat.numel(), -1))
        for n, g in zip(P, gs[1:]):
            grads[n] += g
        pred[s:s + c] = p.detach()
        loss += lc.detach()
        up = ((p - yc) / nb).detach().abs()                          # |d loss / d logit|
        del X, logit, p, lc, gs
        Xa = rows[idx].double().abs().requires_grad_(True)
        la, _ = fwd(A, Xa, M, True, tr)
        ga = torch.autograd.grad(la, [Xa, *A.values()], grad_outputs=up)
        S.index_add_(0, flat, ga[0].reshape(flat.numel(), -1))
        for n, g in zip(A, ga[1:]):
            mass[n] += g
        del Xa, la, ga, tr
    return {"pred": pred, "loss": loss, "grads": grads, "mass": mass, "g_rows": g_rows, "S": S, "S_plain": S_plain, "stats": stats}


def _group(name):
    if "attention" in name:
        return "attention"
    if "interest_evolution" in name:
        return "gru"
    return "tower"


def _worst_ratio(err, bound):
    return float((err / bound.clamp_min(1e-300)).max())


# ---------------------------------------------------------------------------------------------- one checked step
def afm_dw_floor(B, F, D, A):
    """Dense floor (in eps32 of the mass) of the AFM attention parameters.  afm_dw_tc_kernel keeps U = P^T (ds [z > 0])
    and m1 in tensor-core accumulators for the whole kernel, each summing n = B P / parts pair terms (~55 k at C3) in
    fp32, and dW, db and dh are formed from them.  The error of such a long running sum grows with the partial sums it
    adds to -- about sqrt(n) of the mass for terms of random sign, not a constant number of eps32: at C3 it measured
    up to 56 eps32 of the mass (7x the DENSE_EPS floor), so these three take sqrt(n) eps32 (234 at C3)."""
    import ctypes as C
    from deeplearningrecommendationsystem_b200 import _lib
    parts, nbytes = C.c_int32(0), C.c_size_t(0)
    _lib.check(_lib.load().rs_afm_bwd_tc_plan(B, F, D, A, C.byref(parts), C.byref(nbytes)), "rs_afm_bwd_tc_plan")
    assert parts.value > 0
    return (B * (F * (F - 1) // 2) / parts.value) ** 0.5


def run_steps(label, model, tr, inputs, y, table, keys, params, fwd, capture, chunk, lr, guard=None, table_param=None, steps=2,
              floors=None):
    """`steps` steps of Trainer.train_loop on one batch, each checked against `reference` started from the parameters
    and rows the GPU holds before it.  table: the (rows, D) table tensor; keys (B, K): global row of every lookup;
    params: name -> dense parameter; capture(): the masks / stash the step left (dict of (B, ...) tensors); guard:
    sorted untouched rows to keep bit-identical (None: every untouched row); table_param: the table as a parameter
    with a dense .grad (plain torch SGD on the table) or None (fused rows); floors: name -> dense floor in eps32 of the
    mass where it is not DENSE_EPS."""
    from deeplearningrecommendationsystem_b200 import ops
    uniq, inv = torch.unique(keys, return_inverse=True)
    if guard is None:
        keep = torch.ones(table.shape[0], dtype=torch.bool, device=table.device)
        keep[uniq] = False
        guard = keep.nonzero().view(-1)
        del keep
    snap = table[guard].view(torch.int32).clone()
    worst = {"rows": 0.0, "rows_plain_S": 0.0}
    bands = {}
    for step in range(1, steps + 1):
        what = f"{label} step {step}"
        before = table[uniq].clone()
        pbefore = {n: p.detach().clone() for n, p in params.items()}
        tr.train_loop(*inputs, train_rating=y)
        ops.check_status()
        ref = reference(fwd, pbefore, before, inv, y, capture(), chunk)
        np.testing.assert_allclose(tr.predictions_train.detach().reshape(-1).cpu().numpy(), ref["pred"].cpu().numpy(),
                                   rtol=1e-5, atol=1e-6, err_msg=what)
        np.testing.assert_allclose(float(tr.train_loss.detach()), float(ref["loss"]), rtol=1e-5, err_msg=what)
        for name, st in ref["stats"].items():
            b = bands.setdefault(name, {"band": 0, "total": 0, "stash": 0.0})
            b["band"] += st["band"]
            b["total"] += st["total"]
            b["stash"] = max(b["stash"], st["stash"])
            assert st["band"] <= BAND_FRACTION * max(st["total"], 1), f"{what}: {name}: {st['band']} of {st['total']} pre-activations near zero"
        # every touched row
        g64 = ref["g_rows"]
        rows64 = before.double() - lr * g64
        got = table[uniq]
        worst["rows"] = max(worst["rows"], assert_rows_match(got, {"rows": rows64, "grad": g64, "absg": ref["S"]}, lr, what))
        plain = 1e-6 * rows64.abs() + lr * (1e-5 * g64.abs() + 4 * EPS32 * ref["S_plain"])
        worst["rows_plain_S"] = max(worst["rows_plain_S"], _worst_ratio((got.double() - rows64).abs(), plain))
        if table_param is not None:        # plain torch SGD on the table: its dense .grad, touched rows and zero elsewhere
            gt = table_param.grad
            bound = 1e-5 * g64.abs() + 4 * EPS32 * ref["S"]
            err = (gt[uniq].double() - g64).abs()
            assert bool((err <= bound).all()), f"{what}: table .grad off float64 by {_worst_ratio(err, bound):.2f} of the bound"
            assert not bool(gt[guard].any()), f"{what}: untouched rows have a nonzero .grad"
            worst["table_grad"] = max(worst.get("table_grad", 0.0), _worst_ratio(err, bound))
        del before, rows64, got, plain
        # dense parameters: .grad (zero_grad() runs first in train_loop, so it is this step's) and the updated value
        for n, p in params.items():
            g, M = ref["grads"][n], ref["mass"][n]
            bound = 1e-5 * g.abs() + (floors or {}).get(n, DENSE_EPS) * EPS32 * M
            if n.endswith("attention.4.bias"):
                # softmax is shift invariant: d loss / d b2 = 0 analytically, the fp32 sum is rounding noise (kernel tests)
                bound = bound + 1e-5 * float(ref["grads"][n[:-4] + "weight"].abs().max())
            err = (p.grad.double() - g).abs()
            r = _worst_ratio(err, bound)
            assert r <= 1.0, f"{what}: {n}.grad off float64 by {r:.2f} of the bound (max err {float(err.max()):.3e})"
            want = pbefore[n].double() - lr * g
            perr = (p.detach().double() - want).abs()
            pbound = 1e-6 * want.abs() + lr * bound
            pr = _worst_ratio(perr, pbound)
            assert pr <= 1.0, f"{what}: updated {n} off float64 by {pr:.2f} of the bound"
            grp = _group(n)
            worst[grp] = max(worst.get(grp, 0.0), r, pr)
        del ref, pbefore
        same = table[guard].view(torch.int32) == snap
        if not bool(same.all()):
            r = int((~same.all(1)).nonzero()[0])
            raise AssertionError(f"{what}: {int((~same.all(1)).sum())} of {guard.numel()} untouched rows changed, first row {int(guard[r])}")
    band_txt = ", ".join(f"{k} {v['band']}/{v['total']}" for k, v in bands.items() if v["total"])
    stash_txt = ", ".join(f"{k} {v['stash']:.3f}" for k, v in bands.items() if v["stash"])
    return (f"touched rows {uniq.numel()}, untouched checked {guard.numel()}; worst err/bound "
            + ", ".join(f"{k} {v:.2e}" for k, v in worst.items()) + f"; near-zero band {band_txt}"
            + (f"; stash err/bound {stash_txt}" if stash_txt else ""))


# ---------------------------------------------------------------------------------------------- builders
@pytest.fixture
def c3_case(big_case):
    """big_case, and the AFM backward's cached workspace released with the case"""
    yield big_case
    from deeplearningrecommendationsystem_b200 import ops
    ops._afm_ws.clear()


def _dense_params(m):
    return {n: p for n, p in m.named_parameters() if p.requires_grad and not n.endswith("item_embedding.weight")}


def _c3_model(kind):
    from deeplearningrecommendationsystem_b200.nfield import FieldAFM, FieldPNN
    torch.manual_seed(0)           # the nn.Linear layers: two builds are identical
    if kind == "pnn":
        return FieldPNN(C3_CARDS, C3_D, [256, 128, 64, 32], seed=1, device="cuda")
    return FieldAFM(C3_CARDS, C3_D, 64, seed=2, device="cuda")


def _c3_opt(m):
    """FusedRowOptimizer(kind="sgd") over torch SGD for the dense parameters, as bench.py builds it"""
    from deeplearningrecommendationsystem_b200.optim import FusedRowOptimizer
    return FusedRowOptimizer(m, torch.optim.SGD([p for p in m.parameters() if p.requires_grad], lr=C3_LR), lr=C3_LR, kind="sgd")


def _c4_model(kind, dense_tables=False, seed=0):
    from deeplearningrecommendationsystem_b200 import model as M
    torch.manual_seed(seed)
    m = (M.DIN if kind == "din" else M.DIEN)(C4_ITEMS, C4_D).cuda()
    return m if dense_tables else m.fuse_embedding_updates()


def _c4_opt(m, dense_tables=False):
    """bench.py --workload c4: FusedRowOptimizer over torch SGD, or (--dense-tables) torch SGD over everything"""
    from deeplearningrecommendationsystem_b200.optim import FusedRowOptimizer
    if dense_tables:
        return torch.optim.SGD(m.parameters(), lr=C4_LR)
    return FusedRowOptimizer(m, torch.optim.SGD([p for p in m.parameters() if p.requires_grad], lr=C4_LR), lr=C4_LR, kind="sgd")


def c4_batch(seed):
    """zipf history and uniform targets as bench.py draws them; samples pinned to row 0 and row C4_ITEMS - 1"""
    g = torch.Generator(device="cuda").manual_seed(seed)
    hist = zipf_ids(C4_ITEMS, (C4_B, C4_L), g, "cuda")
    tgt = torch.randint(0, C4_ITEMS, (C4_B,), generator=g, device="cuda")
    hist[0], tgt[0], tgt[C4_B // 2] = 0, 0, 0
    hist[1], tgt[1], tgt[C4_B - 1] = C4_ITEMS - 1, C4_ITEMS - 1, C4_ITEMS - 1
    y = (torch.rand(C4_B, 1, generator=g, device="cuda") < 0.3).float()
    return (hist, tgt), y


# ---------------------------------------------------------------------------------------------- C3
@pytest.mark.gpu
@pytest.mark.parametrize("dist", ["uniform", "zipf"])
@pytest.mark.parametrize("kind", ["pnn", "afm"])
def test_c3_step_matches_float64(kind, dist, c3_case, monkeypatch):
    """FieldPNN(CRITEO + [64]*13, 32, [256, 128, 64, 32]) / FieldAFM(same, 32, 64): 33.8 M rows x 32 floats, B = 32768,
    lr 0.05; two steps of Trainer.train_loop on one batch against `reference` with the kernels' ReLU masks."""
    from deeplearningrecommendationsystem_b200 import ops
    from deeplearningrecommendationsystem_b200.trainer import Trainer
    free = need_free(C3_GB)
    ids, y = make_batch(C3_CARDS, dist, seed=(41 if dist == "uniform" else 42), nb=C3_B)
    m = c3_case["model"] = _c3_model(kind)
    tr = c3_case["trainer"] = Trainer(m, torch.nn.BCELoss(), _c3_opt(m))
    cap = c3_case["capture"] = {}
    if kind == "pnn":
        for k, layer in enumerate(m.dnn_network):
            layer.register_forward_hook(lambda mod, inp, out, k=k: cap.__setitem__(f"dnn_network.{k}", out.detach() > 0))
        fwd, chunk, floors = pnn_logit, 4096, None
    else:
        real = ops.afm_bwd

        def afm_bwd(*a, **kw):
            out = real(*a, return_masks=True, **kw)
            assert len(out) == 5, "the C3 AFM backward did not take the tensor-core path"
            cap["attention"] = out[4]
            return out[:4]
        monkeypatch.setattr(ops, "afm_bwd", afm_bwd)
        fwd, chunk = afm_logit, 4096
        f = afm_dw_floor(C3_B, len(C3_CARDS), C3_D, m.attention_W.shape[1])
        floors = {n: f for n in ("attention_W", "attention_b", "attention_h")}
    keys = ids + torch.tensor(m.offsets_host, device="cuda")
    guard, _ = guard_rows(m.cards, m.width, torch.unique(keys), seed=5)
    info = run_steps(f"c3 {kind} {dist}", m, tr, (ids,), y.view(-1, 1), m.weight.data, keys, _dense_params(m), fwd,
                     lambda: dict(cap), chunk, C3_LR, guard=guard, floors=floors)
    c3_case["info"] = f"c3 {kind} {dist}: {free}, {info}"


# ---------------------------------------------------------------------------------------------- C4
@pytest.mark.gpu
@pytest.mark.parametrize("kind,dense_tables", [("din", False), ("dien", False), ("din", True)])
def test_c4_step_matches_float64(kind, dense_tables, big_case, monkeypatch):
    """model.DIN / model.DIEN (1 M items, D = 64) at B = 8192, L = 100, lr 0.01, fused sparse rows
    (fuse_embedding_updates() + FusedRowOptimizer) or, as bench.py --dense-tables, torch SGD on a dense-gradient table"""
    from deeplearningrecommendationsystem_b200 import ops
    from deeplearningrecommendationsystem_b200.trainer import Trainer
    free = need_free(C4_GB)
    ins, y = c4_batch(51 if kind == "din" else 52)
    m = big_case["model"] = _c4_model(kind, dense_tables)
    tr = big_case["trainer"] = Trainer(m, torch.nn.BCELoss(), _c4_opt(m, dense_tables))
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
    emb = m.item_embedding if kind == "din" else m.din.item_embedding
    keys = torch.cat([ins[0], ins[1].unsqueeze(1)], dim=1)
    info = run_steps(f"c4 {kind}{' dense tables' if dense_tables else ''}", m, tr, ins, y, emb.weight.data, keys, _dense_params(m),
                     din_logit if kind == "din" else dien_logit, capture, 2048, C4_LR,
                     table_param=emb.weight if dense_tables else None)
    big_case["info"] = f"c4 {kind}{' dense tables' if dense_tables else ''}: {free}, {info}"


# ---------------------------------------------------------------------------------------------- CPU pin of the reference
def _tiny_field_case(kind):
    from oracle import interactions as OI
    g = torch.Generator().manual_seed(8)
    cards, D, nb = [7, 30, 4, 50, 9, 12], 8, 300
    F = len(cards)
    if kind == "pnn":
        shapes = {"linear1": (16, F * D), "linear2": (16, F * (F - 1) // 2), "dnn_network.0": (12, 16), "dnn_network.1": (6, 12),
                  "output": (1, 6)}
    else:
        shapes = {"output_layer": (1, D)}
    sd = {}
    for n, (o, i) in shapes.items():
        sd[n + ".weight"] = torch.randn(o, i, generator=g, dtype=torch.float64) / i ** 0.5
        sd[n + ".bias"] = torch.randn(o, generator=g, dtype=torch.float64) * 0.1
    if kind == "afm":
        sd.update(attention_W=torch.randn(D, 5, generator=g, dtype=torch.float64) * 0.5,
                  attention_b=torch.randn(5, generator=g, dtype=torch.float64) * 0.1,
                  attention_h=torch.randn(5, 1, generator=g, dtype=torch.float64))
    table = torch.randn(sum(cards), D, generator=g, dtype=torch.float64) * 0.5
    offs = torch.tensor([sum(cards[:k]) for k in range(F)])
    ids = torch.stack([torch.randint(0, c, (nb,), generator=g) for c in cards], dim=1)
    y = (torch.rand(nb, generator=g) < 0.4).double()

    def oracle(sd, E):          # the restatement of test_field_pnn_afm_train_steps, built from oracle.interactions
        if kind == "pnn":
            h = E.flatten(1) @ sd["linear1.weight"].t() + sd["linear1.bias"] + OI.inner_products(E) @ sd["linear2.weight"].t() + sd["linear2.bias"]
            k = 0
            while f"dnn_network.{k}.weight" in sd:
                h = torch.relu(h @ sd[f"dnn_network.{k}.weight"].t() + sd[f"dnn_network.{k}.bias"])
                k += 1
            return torch.sigmoid(h @ sd["output.weight"].t() + sd["output.bias"]).view(-1)
        pooled = OI.afm_pool(E, sd["attention_W"], sd["attention_b"], sd["attention_h"])
        return torch.sigmoid(pooled @ sd["output_layer.weight"].t() + sd["output_layer.bias"]).view(-1)

    E = table[ids + offs]
    if kind == "pnn":
        masks, h = {}, E.flatten(1) @ sd["linear1.weight"].t() + sd["linear1.bias"] + OI.inner_products(E) @ sd["linear2.weight"].t() + sd["linear2.bias"]
        for k in range(2):
            z = h @ sd[f"dnn_network.{k}.weight"].t() + sd[f"dnn_network.{k}.bias"]
            masks[f"dnn_network.{k}"], h = z > 0, torch.relu(z)
    else:
        i, j = OI.pair_index(F)
        masks = {"attention": (E[:, i] * E[:, j]) @ sd["attention_W"] + sd["attention_b"] > 0}
    return sd, table, ids + offs, y, masks, oracle, (pnn_logit if kind == "pnn" else afm_logit)


def _tiny_din_case(kind):
    from oracle import ml100k
    from deeplearningrecommendationsystem_b200 import model as M
    torch.manual_seed(3)
    items, D, L, nb = 60, 8, 7, 200
    m = (M.DIN if kind == "din" else M.DIEN)(items, D).double()
    with torch.no_grad():                                  # biases away from zero so that the masks are not all-or-nothing
        for n, p in m.named_parameters():
            if n.endswith("bias"):
                p.normal_(0.0, 0.2)
    sd = {k: v.detach().clone() for k, v in m.state_dict().items()}
    g = torch.Generator().manual_seed(9)
    hist = torch.randint(0, items, (nb, L), generator=g)
    tgt = torch.randint(0, items, (nb,), generator=g)
    y = (torch.rand(nb, generator=g) < 0.4).double()
    pfx = "" if kind == "din" else "din."
    tab = sd[pfx + "item_embedding.weight"]
    h, t = tab[hist], tab[tgt]
    x = torch.cat([h, h - t.unsqueeze(1), t.unsqueeze(1).expand_as(h)], dim=-1)
    z0 = x @ sd[pfx + "attention.0.weight"].t() + sd[pfx + "attention.0.bias"]
    z1 = torch.relu(z0) @ sd[pfx + "attention.2.weight"].t() + sd[pfx + "attention.2.bias"]
    s = torch.relu(z1) @ sd[pfx + "attention.4.weight"].t() + sd[pfx + "attention.4.bias"]
    w = torch.softmax(s.squeeze(-1), dim=-1)
    if kind == "din":
        f = torch.cat([(h * w.unsqueeze(-1)).sum(1), t], dim=1)
    else:
        with torch.no_grad():
            f = torch.cat([m.interest_evolution(h * w.unsqueeze(-1))[1][-1], t], dim=1)
    a = f @ sd["fc.0.weight"].t() + sd["fc.0.bias"]
    b = torch.relu(a) @ sd["fc.2.weight"].t() + sd["fc.2.bias"]
    masks = {"act0": z0 > 0, "act1": z1 > 0, "act0_val": torch.relu(z0), "act1_val": torch.relu(z1), "attw_val": w,
             "fc.1": a > 0, "fc.3": b > 0}
    oracle = (lambda sd, hh, tt: ml100k.din(sd, hh, tt).view(-1)) if kind == "din" else (lambda sd, hh, tt: ml100k.dien(sd, hh, tt).view(-1))
    return sd, tab, torch.cat([hist, tgt.unsqueeze(1)], dim=1), hist, tgt, y, masks, oracle, (din_logit if kind == "din" else dien_logit)


@pytest.mark.parametrize("kind", ["pnn", "afm", "din", "dien"])
def test_reference_matches_the_oracle_restatements(kind):
    """`reference` with masks = (z > 0), in float64 on the CPU, against the restatements it replaces: the PNN / AFM one
    of test_field_pnn_afm_train_steps (oracle.interactions) and oracle.ml100k.din / dien on a state dict -- predictions,
    loss, every dense gradient and the summed row gradient to 1e-12; the mass pass bounds every gradient."""
    from oracle import interactions as OI
    if kind in ("pnn", "afm"):
        sd, table, keys, y, masks, oracle, fwd = _tiny_field_case(kind)
        leaves = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
        tab = table.clone().requires_grad_(True)
        pred = oracle(leaves, tab[keys])
        params = sd
    else:
        sd, table, keys, hist, tgt, y, masks, oracle, fwd = _tiny_din_case(kind)
        pfx = "" if kind == "din" else "din."
        leaves = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
        tab = leaves[pfx + "item_embedding.weight"]
        pred = oracle(leaves, hist, tgt)
        params = {k: v for k, v in sd.items() if not k.endswith("item_embedding.weight")}
    loss = OI.bce(pred, y)
    names = [k for k in params]
    got = torch.autograd.grad(loss, [tab] + [leaves[k] for k in names])
    uniq, inv = torch.unique(keys, return_inverse=True)
    ref = reference(fwd, params, table[uniq], inv, y, masks, chunk=70)
    close = lambda a, b, what: np.testing.assert_allclose(a.detach().numpy(), b.detach().numpy(), rtol=1e-12, atol=1e-15, err_msg=what)  # noqa: E731
    close(ref["pred"], pred, "pred")
    close(ref["loss"], loss, "loss")
    close(ref["g_rows"], got[0][uniq], "rows")
    untouched = torch.ones(table.shape[0], dtype=torch.bool)
    untouched[uniq] = False
    assert not bool(got[0][untouched].any())
    for k, g in zip(names, got[1:]):
        close(ref["grads"][k], g, k)
        assert bool((ref["mass"][k] >= g.abs() * (1 - 1e-12)).all()), k
    assert bool((ref["S"] >= ref["S_plain"] * (1 - 1e-12)).all()) and bool((ref["S_plain"] >= ref["g_rows"].abs() * (1 - 1e-12)).all())
    for name, st in ref["stats"].items():
        assert st["total"] == 0 or st["band"] < st["total"], name


# ---------------------------------------------------------------------------------------------- graphed == eager
@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["pnn", "afm", "din", "dien"])
def test_graphed_step_equals_eager_at_benchmark_shapes(kind, c3_case):
    """GraphedTrainStep(warmup=1) -- what bench.py times -- against eager Trainer.train_loop on two identical models
    over the same three batches: bit-identical predictions, losses, parameters and tables"""
    from deeplearningrecommendationsystem_b200.graph import GraphedTrainStep
    from deeplearningrecommendationsystem_b200.trainer import Trainer
    free = need_free(2 * C3_GB if kind in ("pnn", "afm") else C4_GB)
    if kind in ("pnn", "afm"):
        m1, m2 = _c3_model(kind), _c3_model(kind)
        o1, o2 = _c3_opt(m1), _c3_opt(m2)
        batches = [make_batch(C3_CARDS, "zipf" if k == 1 else "uniform", seed=60 + k, nb=C3_B) for k in range(3)]
        batches = [((ids,), y.view(-1, 1)) for ids, y in batches]
        tables = lambda m: [m.weight]                                     # noqa: E731
    else:
        m1, m2 = _c4_model(kind, seed=4), _c4_model(kind, seed=4)
        o1, o2 = _c4_opt(m1), _c4_opt(m2)
        batches = [c4_batch(70 + k) for k in range(3)]
        tables = lambda m: [(m.item_embedding if kind == "din" else m.din.item_embedding).weight]   # noqa: E731
    c3_case["model"] = (m1, m2)
    assert all(torch.equal(a, b) for a, b in zip(tables(m1), tables(m2)))
    tr = Trainer(m1, torch.nn.BCELoss(), o1)
    gs = GraphedTrainStep(m2, torch.nn.BCELoss(), o2, warmup=1)
    for k, (ins, y) in enumerate(batches):
        tr.train_loop(*ins, train_rating=y)
        pred, loss = gs(*ins, rating=y)
        assert torch.equal(pred, tr.predictions_train), f"step {k}: predictions differ"
        assert torch.equal(loss, tr.train_loss), f"step {k}: losses differ"
    assert gs.graph is not None
    for (n, a), (_, b) in zip(m1.named_parameters(), m2.named_parameters()):
        assert torch.equal(a, b), f"{n} differs between the graphed and the eager step"
    for a, b in zip(tables(m1), tables(m2)):
        assert torch.equal(a, b), "table differs between the graphed and the eager step"
    c3_case["info"] = f"graphed == eager {kind}: {free}"
    del gs, tr
    gc.collect()


# ---------------------------------------------------------------------------------------------- captured AFM workspace
@pytest.mark.gpu
def test_captured_afm_backward_keeps_its_workspace():
    """ops.afm_bwd caches one workspace per device and drops it for a larger shape.  A captured step must not run on
    that cached block: after an eager backward at a larger batch has replaced it, the block belongs to whatever tensor
    the allocator hands it to next (here a sentinel), and every replay would write ds, mask bits and dP into it."""
    from deeplearningrecommendationsystem_b200 import ops
    from deeplearningrecommendationsystem_b200.graph import GraphedTrainStep
    from deeplearningrecommendationsystem_b200.nfield import FieldAFM
    from deeplearningrecommendationsystem_b200.optim import FusedRowOptimizer
    from deeplearningrecommendationsystem_b200.trainer import Trainer
    cards, D, A, nb, lr = [40 + 13 * k for k in range(17)], 16, 32, 4096, 0.1     # 136 pairs: the tensor-core backward
    dev = torch.device("cuda", torch.cuda.current_device())
    ops._afm_ws.clear()

    def opt_for(m):
        return FusedRowOptimizer(m, torch.optim.SGD([p for p in m.parameters() if p.requires_grad], lr=lr), lr=lr)
    def build():
        torch.manual_seed(0)       # the output layer: two builds are identical
        return FieldAFM(cards, D, A, seed=3, device="cuda")
    m1, m2 = build(), build()
    tr = Trainer(m1, torch.nn.BCELoss(), opt_for(m1))
    gs = GraphedTrainStep(m2, torch.nn.BCELoss(), opt_for(m2), warmup=1)
    g = torch.Generator(device="cuda").manual_seed(13)

    def batch():
        ids = torch.stack([torch.randint(0, c, (nb,), generator=g, device="cuda") for c in cards], dim=1)
        return ids, (torch.rand(nb, 1, generator=g, device="cuda") < 0.3).float()

    def step(ids, y):
        tr.train_loop(ids, train_rating=y)
        pred, loss = gs(ids, rating=y)
        assert torch.equal(pred, tr.predictions_train) and torch.equal(loss, tr.train_loss)
    step(*batch())                                 # eager: the workspace is allocated and cached
    step(*batch())                                 # capture + first replay
    assert gs.graph is not None
    old = ops._afm_ws[dev]
    old_ptr, old_n = old.data_ptr(), old.numel()
    del old
    # an eager backward at twice the batch replaces the cached workspace ...
    E = torch.randn(2 * nb, len(cards), D, generator=g, device="cuda") * 0.3
    W, b, h = m1.attention_W.detach(), m1.attention_b.detach(), m1.attention_h.detach()
    _, attw = ops.afm_fwd(E, W, b, h)
    ops.afm_bwd(E, W, b, h, attw, torch.randn(2 * nb, D, generator=g, device="cuda"))
    assert ops._afm_ws[dev].numel() > old_n
    # ... and the block it held goes to the next tensor of its size
    sentinel = torch.full((old_n,), 0x5A, dtype=torch.uint8, device="cuda")
    assert sentinel.data_ptr() == old_ptr, "the allocator placed the sentinel elsewhere: this test cannot see the hazard"
    step(*batch())                                 # replay
    torch.cuda.synchronize()
    changed = int((sentinel != 0x5A).sum())
    assert changed == 0, f"the graph replay wrote {changed} bytes into memory the AFM workspace cache had released"
    for (n, a), (_, b_) in zip(m1.named_parameters(), m2.named_parameters()):
        assert torch.equal(a, b_), f"{n} differs between the graphed and the eager step"
