"""The PNN paper's outer-product layer (OPNN, sum pooling): rs_pnn_outer_fwd / rs_pnn_outer_bwd and
FieldPNN(product="outer").  The reference has no such layer (its "out" mode collapses the batch, model.PNN), so parity
is unpinned by the reference: the kernels are pinned to the float64 restatement `restate`, which is itself checked
against torch autograd of the literal formula Linear(D*D, H0)(vec(s s^T)) on the CPU.

Bound (the DENSE_EPS rule of test_c3_c4_shapes_gpu): |x - x64| <= 1e-5 |x64| + 8 eps32 mass, mass = the same
contraction over absolute values."""
import ctypes as C
import gc

import numpy as np
import pytest
import torch

from test_c3_c4_shapes_gpu import (C3_B, C3_CARDS, C3_D, C3_GB, C3_LR, DENSE_EPS, _c3_opt, _dense_params, _lin, c3_case,  # noqa: F401
                                   need_free, reference, run_steps)
from test_full_scale_gpu import EPS32, big_case, guard_rows, make_batch  # noqa: F401


# ---------------------------------------------------------------------------------------------- float64 restatement
def restate(E, W, b, g):
    """lp, dS, dW, db of the layer for E (B, F, D), W (H0, D*D), b (H0), g = d loss / d lp (B, H0), and the mass of each
    (the same contractions over absolute values).  Any dtype; call it with float64."""
    B, F, D = E.shape
    H0 = W.shape[0]

    def layer(E, W, b, g):
        s = E.sum(1)
        W3 = W.reshape(H0, D, D)
        p = (s.unsqueeze(2) * s.unsqueeze(1)).reshape(B, D * D)
        lp = p @ W.t() + b
        dS = ((g @ (W3 + W3.transpose(1, 2)).reshape(H0, D * D)).reshape(B, D, D) * s.unsqueeze(1)).sum(2)
        return {"S": s, "lp": lp, "dS": dS, "dW": g.t() @ p, "db": g.sum(0)}
    return layer(E, W, b, g), layer(E.abs(), W.abs(), b.abs(), g.abs())


def _inputs(B, F, D, H0, seed, device):
    gen = torch.Generator(device="cpu").manual_seed(seed)
    E = torch.randn(B, F, D, generator=gen) * (0.5 / F ** 0.5)
    W = torch.randn(H0, D * D, generator=gen) / D          # not symmetric in (i, j)
    b = torch.randn(H0, generator=gen) * 0.1
    g = torch.randn(B, H0, generator=gen) * 1e-3
    if B > 2:
        E[B // 2] = 0.0                                      # an all-zero sample: lp = bias, dS = 0
    return [t.to(device) for t in (E, W, b, g)]


def _within(name, got, want, mass):
    err = (got.double() - want).abs()
    bound = 1e-5 * want.abs() + DENSE_EPS * EPS32 * mass
    r = float((err / bound.clamp_min(1e-300)).max()) if err.numel() else 0.0
    assert r <= 1.0, f"{name}: off float64 by {r:.2f} of the bound (max err {float(err.max()):.3e})"


# ---------------------------------------------------------------------------------------------- CPU
def test_restatement_matches_autograd_of_the_formula():
    """restate() == autograd of Linear(D*D, H0)(vec(s s^T)), s = sum_f e_f, in float64"""
    B, F, D, H0 = 37, 3, 8, 16
    E, W, b, g = (t.double() for t in _inputs(B, F, D, H0, 1, "cpu"))
    lin = torch.nn.Linear(D * D, H0).double()
    with torch.no_grad():
        lin.weight.copy_(W)
        lin.bias.copy_(b)
    Ev = E.clone().requires_grad_(True)
    s = Ev.sum(1)
    lp = lin((s.unsqueeze(2) * s.unsqueeze(1)).reshape(B, D * D))
    (lp * g).sum().backward()
    r, m = restate(E, W, b, g)
    close = lambda a, b_: np.testing.assert_allclose(a.detach().numpy(), b_.detach().numpy(), rtol=1e-12, atol=1e-15)  # noqa: E731
    close(r["lp"], lp)
    for f in range(F):
        close(r["dS"], Ev.grad[:, f])
    close(r["dW"], lin.weight.grad)
    close(r["db"], lin.bias.grad)
    assert bool((r["lp"][B // 2] == b).all()) and not bool(r["dS"][B // 2].any())
    for k in r:
        assert bool((m[k] >= r[k].abs() * (1 - 1e-12)).all()), k


def test_abi_rejects_unsupported_shapes_and_null_pointers():
    from deeplearningrecommendationsystem_b200 import _lib
    lib = _lib.load()
    f, b = C.c_size_t(0), C.c_size_t(0)
    assert lib.rs_pnn_outer_ws_bytes(1000, 32, 256, C.byref(f), C.byref(b)) == 0 and f.value == 2 * 256 * 32 * 32 * 4
    for D, H0, limit in ((24, 256, b"D must be 16, 32 or 64"), (8, 64, b"D must be 16, 32 or 64"),
                         (32, 40, b"H0 must be a multiple of 16 in [16, 512]"), (32, 528, b"H0 must be a multiple of 16 in [16, 512]"),
                         (32, 0, b"H0 must be a multiple of 16 in [16, 512]")):
        assert lib.rs_pnn_outer_ws_bytes(10, D, H0, C.byref(f), C.byref(b)) == -4                 # RS_E_UNSUPPORTED
        assert limit in lib.rs_last_error()
        p = C.c_void_p(16)                                                                          # never dereferenced
        assert lib.rs_pnn_outer_fwd(p, 10, 2, D, H0, p, p, p, p, p, 1 << 30, None) == -4
        assert limit in lib.rs_last_error() and b"rs_pnn_outer_fwd" in lib.rs_last_error()
        assert lib.rs_pnn_outer_bwd(p, p, 10, D, H0, p, p, p, p, p, 1 << 30, None) == -4
        assert limit in lib.rs_last_error() and b"rs_pnn_outer_bwd" in lib.rs_last_error()
    assert lib.rs_pnn_outer_fwd(None, 10, 2, 32, 256, None, None, None, None, None, 0, None) == -1      # RS_E_ARG
    assert b"null pointer" in lib.rs_last_error()
    assert lib.rs_pnn_outer_bwd(None, None, 10, 32, 256, None, None, None, None, None, 0, None) == -1
    assert b"null pointer" in lib.rs_last_error()
    assert lib.rs_pnn_outer_ws_bytes(10, 32, 256, None, None) == -1


def test_field_pnn_outer_builds_on_cpu_and_rejects_unknown_products():
    from deeplearningrecommendationsystem_b200.nfield import FieldPNN
    m = FieldPNN([5, 7, 9], 16, [32, 8], product="outer")
    assert tuple(m.state_dict()["linear2.weight"].shape) == (32, 256)
    assert tuple(FieldPNN([5, 7, 9], 16, [32, 8]).state_dict()["linear2.weight"].shape) == (32, 3)
    with pytest.raises(ValueError, match="inner"):
        FieldPNN([5, 7, 9], 16, [32, 8], product="both")


# ---------------------------------------------------------------------------------------------- GPU: kernels vs float64
def _cases():
    out = []
    for D in (16, 32, 64):
        for k, B in enumerate((1, 127, 128, 129, 1000, 32768)):
            for H0 in (16, 512):
                out.append((D, H0, (1, 2, 39)[(k + H0 // 512) % 3], B))
    out += [(32, 256, 39, 32768), (16, 48, 2, 1000), (64, 144, 39, 129)]
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("D,H0,F,B", _cases())
def test_kernels_match_float64(D, H0, F, B):
    """lp, S, dS, dW, db against `restate` in float64; a second run of forward and backward is bit-identical"""
    from deeplearningrecommendationsystem_b200 import ops
    E, W, b, g = _inputs(B, F, D, H0, seed=D * 1000 + H0 + B, device="cuda")
    lp, S = ops.pnn_outer_fwd(E, W, b)
    dS, dW, db = ops.pnn_outer_bwd(S, g, W)
    r, m = restate(E.double(), W.double(), b.double(), g.double())
    for name, got in (("S", S), ("lp", lp), ("dS", dS), ("dW", dW), ("db", db)):
        _within(f"D={D} H0={H0} F={F} B={B} {name}", got, r[name], m[name])
    if B > 2:
        assert torch.equal(lp[B // 2], b), "an all-zero sample must give lp = bias"
        assert not bool(dS[B // 2].any()), "an all-zero sample must give dS = 0"
    lp2, S2 = ops.pnn_outer_fwd(E, W, b)
    dS2, dW2, db2 = ops.pnn_outer_bwd(S2, g, W)
    for a, c in ((lp, lp2), (S, S2), (dS, dS2), (dW, dW2), (db, db2)):
        assert torch.equal(a, c), "two runs differ"


@pytest.mark.gpu
def test_empty_batch():
    from deeplearningrecommendationsystem_b200 import ops
    E, W, b, g = _inputs(0, 3, 32, 64, 0, "cuda")
    lp, S = ops.pnn_outer_fwd(E, W, b)
    dS, dW, db = ops.pnn_outer_bwd(S, g, W)
    assert lp.shape == (0, 64) and S.shape == (0, 32) and dS.shape == (0, 32)
    assert not bool(dW.any()) and not bool(db.any())


@pytest.mark.gpu
def test_ops_raise_with_the_limit():
    from deeplearningrecommendationsystem_b200 import ops
    E, W, b, _ = _inputs(10, 2, 32, 40, 0, "cuda")
    with pytest.raises(RuntimeError, match=r"H0 must be a multiple of 16 in \[16, 512\]"):
        ops.pnn_outer_fwd(E, W, b)
    E, W, b, _ = _inputs(10, 2, 8, 32, 0, "cuda")
    with pytest.raises(RuntimeError, match="D must be 16, 32 or 64"):
        ops.pnn_outer_fwd(E, W, b)


# ---------------------------------------------------------------------------------------------- GPU: small model
def _tower(P, h):
    k = 0
    while f"dnn_network.{k}.weight" in P:
        h = torch.relu(_lin(h, P, f"dnn_network.{k}"))
        k += 1
    return torch.sigmoid(_lin(h, P, "output")).view(-1)


@pytest.mark.gpu
@pytest.mark.parametrize("kind,wd", [("sgd", 0.0), ("adam", 1e-2)])
def test_small_field_pnn_outer_train_steps(kind, wd):
    """FieldPNN(product="outer") on a small table with heavy duplicates, Trainer.train_loop + FusedRowOptimizer (lazy row
    SGD / Adam with weight decay, torch SGD / Adam on the dense layers), two steps against float64: predictions, loss,
    every dense .grad and parameter, every touched row; untouched rows bit-identical; eval() + no_grad() inference."""
    from deeplearningrecommendationsystem_b200.nfield import FieldPNN
    from deeplearningrecommendationsystem_b200.optim import FusedRowOptimizer
    from deeplearningrecommendationsystem_b200.trainer import Trainer
    from oracle import interactions as OI
    from oracle import optim as OO
    cards, D, hidden, B, lr = [7, 300, 40, 1000, 5, 64, 12], 16, [32, 16, 8], 600, (0.2 if kind == "sgd" else 0.01)
    gen = torch.Generator().manual_seed(4)
    ids = torch.stack([(torch.rand(B, generator=gen) ** 3 * c).long().clamp_(max=c - 1) for c in cards], dim=1)
    y = (torch.rand(B, 1, generator=gen) < 0.4).float()
    torch.manual_seed(0)
    m = FieldPNN(cards, D, hidden, seed=2, device="cuda", product="outer")
    assert tuple(m.state_dict()["linear2.weight"].shape) == (hidden[0], D * D)
    dense = [p for p in m.parameters() if p.requires_grad]
    dopt = torch.optim.SGD(dense, lr=lr) if kind == "sgd" else torch.optim.Adam(dense, lr=lr, weight_decay=wd)
    tr = Trainer(m, torch.nn.BCELoss(), FusedRowOptimizer(m, dopt, lr=lr, kind=kind, weight_decay=wd))
    names = [n for n, p in m.named_parameters() if p.requires_grad]
    P = {n: p.detach().double().cpu().clone() for n, p in m.named_parameters() if p.requires_grad}
    table = m.weight.detach().double().cpu().clone()
    tm, tv = torch.zeros_like(table), torch.zeros_like(table)
    pm = {n: torch.zeros_like(p) for n, p in P.items()}
    pv = {n: torch.zeros_like(p) for n, p in P.items()}
    keys = ids + torch.tensor(m.offsets_host)
    untouched = torch.ones(table.shape[0], dtype=torch.bool)
    untouched[keys.unique()] = False
    snap = m.weight.detach()[untouched.cuda()].clone()
    for step in range(1, 3):
        tr.train_loop(ids.cuda(), train_rating=y.cuda())
        leaves = {n: p.clone().requires_grad_(True) for n, p in P.items()}
        tab = table.clone().requires_grad_(True)
        E = tab[keys]
        s = E.sum(1)
        p = (s.unsqueeze(2) * s.unsqueeze(1)).reshape(B, D * D)
        h = _lin(E.flatten(1), leaves, "linear1") + _lin(p, leaves, "linear2")
        pred = _tower(leaves, h)
        loss = OI.bce(pred, y.view(-1).double())
        grads = torch.autograd.grad(loss, [tab] + [leaves[n] for n in names])
        what = f"{kind} step {step}"
        np.testing.assert_allclose(tr.predictions_train.detach().cpu().view(-1).numpy(), pred.detach().numpy(), rtol=1e-5, atol=1e-6,
                                   err_msg=what)
        np.testing.assert_allclose(tr.train_loss.item(), loss.item(), rtol=1e-5, err_msg=what)
        for n, gr in zip(names, grads[1:]):
            got = dict(m.named_parameters())[n].grad.detach().cpu().double()
            np.testing.assert_allclose(got.numpy(), gr.numpy(), rtol=1e-4, atol=1e-5 * float(gr.abs().max()), err_msg=f"{what}: {n}.grad")
        with torch.no_grad():
            rows = keys.unique()
            if kind == "sgd":
                table[rows] -= lr * grads[0][rows]
                for n, gr in zip(names, grads[1:]):
                    P[n] -= lr * gr
            else:
                OO.adam_rows(table, tm, tv, rows, grads[0][rows], step, lr=lr, wd=wd)
                for n, gr in zip(names, grads[1:]):
                    P[n], pm[n], pv[n] = OO.adam_dense(P[n], gr, pm[n], pv[n], step, lr=lr, wd=wd)
        atol = 2e-6 if kind == "sgd" else 2e-4
        np.testing.assert_allclose(m.weight.detach()[rows.cuda()].cpu().numpy(), table[rows].numpy(), rtol=1e-5, atol=atol, err_msg=f"{what}: rows")
        for n in names:
            np.testing.assert_allclose(dict(m.named_parameters())[n].detach().cpu().numpy(), P[n].numpy(), rtol=1e-5, atol=atol,
                                       err_msg=f"{what}: {n}")
        assert torch.equal(m.weight.detach()[untouched.cuda()], snap), f"{what}: untouched rows changed"
    m.eval()
    with torch.no_grad():
        out = m(ids.cuda())
        E = table[keys]
        s = E.sum(1)
        want = _tower(P, _lin(E.flatten(1), P, "linear1") + _lin((s.unsqueeze(2) * s.unsqueeze(1)).reshape(B, D * D), P, "linear2"))
    np.testing.assert_allclose(out.cpu().view(-1).numpy(), want.numpy(), rtol=1e-5, atol=1e-6)


# ---------------------------------------------------------------------------------------------- GPU: the C3 step
def pnn_outer_logit(P, X, M, am, tr):
    """FieldPNN(product="outer"): X (c, F, D) rows of the lookups; M: the dnn_network masks"""
    c, F, D = X.shape
    s = X.sum(1)
    h = _lin(X.reshape(c, F * D), P, "linear1") + _lin((s.unsqueeze(2) * s.unsqueeze(1)).reshape(c, D * D), P, "linear2")
    checks, k = [], 0
    from test_c3_c4_shapes_gpu import _lin_mass
    while f"dnn_network.{k}.weight" in P:
        name = f"dnn_network.{k}"
        z = _lin(h, P, name)
        if not am:
            checks.append((name, z.detach(), _lin_mass(h, P, name), M[name], None))
        h = z * M[name]
        k += 1
    return _lin(h, P, "output").view(-1), checks


def _c3_outer_model():
    from deeplearningrecommendationsystem_b200.nfield import FieldPNN
    torch.manual_seed(0)
    return FieldPNN(C3_CARDS, C3_D, [256, 128, 64, 32], seed=1, device="cuda", product="outer")


@pytest.mark.gpu
@pytest.mark.parametrize("dist", ["uniform", "zipf"])
def test_c3_outer_step_matches_float64(dist, c3_case):
    """FieldPNN(CRITEO + [64]*13, 32, [256, 128, 64, 32], product="outer") at B = 32768, two steps of Trainer.train_loop
    against `reference` with the tower's ReLU masks borrowed through forward hooks"""
    from deeplearningrecommendationsystem_b200.trainer import Trainer
    free = need_free(C3_GB)
    ids, y = make_batch(C3_CARDS, dist, seed=(43 if dist == "uniform" else 44), nb=C3_B)
    m = c3_case["model"] = _c3_outer_model()
    tr = c3_case["trainer"] = Trainer(m, torch.nn.BCELoss(), _c3_opt(m))
    cap = c3_case["capture"] = {}
    for k, layer in enumerate(m.dnn_network):
        layer.register_forward_hook(lambda mod, inp, out, k=k: cap.__setitem__(f"dnn_network.{k}", out.detach() > 0))
    keys = ids + torch.tensor(m.offsets_host, device="cuda")
    guard, _ = guard_rows(m.cards, m.width, torch.unique(keys), seed=5)
    info = run_steps(f"c3 pnn outer {dist}", m, tr, (ids,), y.view(-1, 1), m.weight.data, keys, _dense_params(m), pnn_outer_logit,
                     lambda: dict(cap), 4096, C3_LR, guard=guard)
    c3_case["info"] = f"c3 pnn outer {dist}: {free}, {info}"


@pytest.mark.gpu
def test_c3_outer_graphed_step_equals_eager(c3_case):
    """GraphedTrainStep(warmup=1) against eager Trainer.train_loop at the C3 shape, bit for bit, over three batches.  Before
    the last replay an eager forward + backward at twice the batch runs and its tensors are freed; the replay must not
    write into that released memory (the captured workspace is the graph's own) and must still equal the eager step."""
    from deeplearningrecommendationsystem_b200 import ops
    from deeplearningrecommendationsystem_b200.graph import GraphedTrainStep
    from deeplearningrecommendationsystem_b200.trainer import Trainer
    free = need_free(2 * C3_GB)
    m1, m2 = _c3_outer_model(), _c3_outer_model()
    c3_case["model"] = (m1, m2)
    assert torch.equal(m1.weight, m2.weight)
    tr = Trainer(m1, torch.nn.BCELoss(), _c3_opt(m1))
    gs = GraphedTrainStep(m2, torch.nn.BCELoss(), _c3_opt(m2), warmup=1)
    batches = [make_batch(C3_CARDS, "zipf" if k == 1 else "uniform", seed=80 + k, nb=C3_B) for k in range(3)]
    sentinels = []
    for k, (ids, y) in enumerate(batches):
        if k == 2:
            assert gs.graph is not None
            E, W, b, g = _inputs(2 * C3_B, len(C3_CARDS), C3_D, 256, 9, "cuda")
            lp, S = ops.pnn_outer_fwd(E, W, b)
            outs = ops.pnn_outer_bwd(S, g, W)
            sizes = [t.numel() for t in (lp, S, *outs)]
            del lp, S, outs, E, g
            torch.cuda.synchronize()
            sentinels = [torch.full((n,), 7.0, device="cuda") for n in sizes]
        tr.train_loop(ids, train_rating=y.view(-1, 1))
        pred, loss = gs(ids, rating=y.view(-1, 1))
        assert torch.equal(pred, tr.predictions_train), f"step {k}: predictions differ"
        assert torch.equal(loss, tr.train_loss), f"step {k}: losses differ"
    torch.cuda.synchronize()
    assert all(bool((t == 7.0).all()) for t in sentinels), "the replay wrote into memory freed by the larger eager call"
    for (n, a), (_, c) in zip(m1.named_parameters(), m2.named_parameters()):
        assert torch.equal(a, c), f"{n} differs between the graphed and the eager step"
    assert torch.equal(m1.weight, m2.weight), "table differs between the graphed and the eager step"
    c3_case["info"] = f"graphed == eager pnn outer: {free}"
    del gs, tr
    gc.collect()
