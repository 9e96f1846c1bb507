"""Adam and weight decay on the replicated small tables of the hybrid multi-GPU placement (rs_mark_rows +
rs_replica_update), on ONE GPU with virtual ranks (dist.ThreadFabric, as in test_shard_gpu.py).

The replicated tables take the lazy row update of the single-GPU FusedRowOptimizer: only rows that some rank's batch
touched step, with the row-update kernels' arithmetic (upd_sgd / adam1).  The kernel is checked bit for bit against
rs_segment_update fed the rank-ordered sum, and the hybrid model against the single-GPU step on the concatenated batch.
"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
CARDS = [3, 50, 7, 1000, 24, 12, 301, 5]
C2_CAPPED = [min(c, 2000) for c in [1460, 583, 10131227, 2202608, 305, 24, 12517, 633, 3, 93145, 5683, 8351593, 3194, 27, 14992,
                                    5461306, 10, 5652, 2173, 4, 7046547, 18, 15, 286181, 105, 142572]]
ADAM_LR, SGD_LR, WD = 0.01, 0.5, 1e-2


def _ops():
    from deeplearningrecommendationsystem_b200 import ops
    return ops


def _rank_sum(grads):
    acc = torch.zeros_like(grads[0])
    for x in grads:
        acc = acc + x                                   # rank order, fp32: the kernel's order
    return acc


def _reference_update(ops, w, m, v, rows_hit, gsum, kind, lr, wd, step):
    """rs_segment_update on (w, m, v) with one lookup per touched row carrying the summed gradient"""
    if rows_hit.numel() == 0:
        return
    W = w.shape[1]
    segs = ops.dedup_sort(rows_hit.cuda(), 1, None, w.shape[0], max_width=W, reuse_workspace=False)
    dense = gsum[rows_hit].contiguous().cuda()
    if kind == "sgd":
        ops.segment_update(segs, ops.RS_UPD_SGD, W, 1, dense=dense, table=w, lr=lr, wd=wd)
    else:
        ops.segment_update(segs, ops.RS_UPD_ADAM, W, 1, dense=dense, table=w, m=m, v=v, lr=lr, wd=wd, step=step)


def _flags(world, rows, step):
    """per-rank touched flags: each row falls in one class, the class rotating with the step -- untouched, touched by
    exactly rank r (each r, owner of the row's slice or not), touched by every rank, touched by every rank with an all-zero
    gradient.  Returns (flags (world, rows) uint8, rows whose gradient must be zero)."""
    ncls = world + 3
    cls = (torch.arange(rows) * 7 + step * 3) % ncls
    flags = torch.zeros(world, rows, dtype=torch.uint8)
    for r in range(world):
        flags[r] = ((cls == 1 + r) | (cls >= world + 1)).to(torch.uint8)
    return flags, (cls == world + 2)


@pytest.mark.parametrize("world,rows,width", [(1, 37, 16), (2, 300, 16), (3, 47, 416), (8, 5, 16), (8, 1, 4)])
@pytest.mark.parametrize("kind,steps", [("sgd", 2), ("adam", 3)])
@pytest.mark.parametrize("wd", [0.0, WD])
def test_replica_update_equals_row_update(world, rows, width, kind, steps, wd):
    """rs_replica_update run by every rank in turn == rs_segment_update on the rank-ordered sum over the flagged rows, bit
    for bit (w, m, v); replicas stay bit-identical; unflagged rows keep their bits although their gradients are nonzero."""
    ops = _ops()
    lr = SGD_LR if kind == "sgd" else ADAM_LR
    g = torch.Generator().manual_seed(world * 1000 + rows + width)
    numel = rows * width
    w0 = torch.randn(rows, width, generator=g)
    W = [w0.clone().cuda() for _ in range(world)]
    ref_w = w0.clone().cuda()
    ref_m, ref_v = torch.zeros_like(ref_w), torch.zeros_like(ref_w)
    bounds = [ops.replica_slice(numel, world, r) for r in range(world)]
    ms = [torch.zeros(hi - lo, device="cuda") for lo, hi in bounds]
    vs = [torch.zeros(hi - lo, device="cuda") for lo, hi in bounds]
    for step in range(1, steps + 1):
        flags, zero_rows = _flags(world, rows, step)
        grads = [torch.randn(rows, width, generator=g) for _ in range(world)]
        for x in grads:
            x[zero_rows] = 0.0
        G = [x.cuda() for x in grads]
        T = [f.cuda() for f in flags]
        before = [t.clone() for t in W], torch.cat(ms).clone(), torch.cat(vs).clone()
        for r in range(world):
            ops.replica_update([t.data_ptr() for t in W], [t.data_ptr() for t in G], [t.data_ptr() for t in T], numel, width, world,
                               r, kind, lr, wd, m=ms[r], v=vs[r], step=step)
        hit = flags.bool().any(0)
        rows_hit = torch.nonzero(hit).view(-1)
        _reference_update(ops, ref_w, ref_m, ref_v, rows_hit, _rank_sum(grads), kind, lr, wd, step)
        torch.cuda.synchronize()
        for r in range(world):
            assert torch.equal(W[r], W[0]), f"replica {r} differs"
        assert torch.equal(W[0], ref_w), f"step {step}: w differs from the row-update kernel"
        miss = (~hit).cuda()
        assert torch.equal(W[0][miss], before[0][0][miss]), "an untouched row moved"
        if kind == "adam":
            assert torch.equal(torch.cat(ms), ref_m.view(-1)), f"step {step}: m differs"
            assert torch.equal(torch.cat(vs), ref_v.view(-1)), f"step {step}: v differs"
            miss_el = miss.view(-1, 1).expand(rows, width).reshape(-1)
            assert torch.equal(torch.cat(ms)[miss_el], before[1][miss_el]) and torch.equal(torch.cat(vs)[miss_el], before[2][miss_el])
    ops.check_status()


def test_replica_update_refuses_grad_mode_and_bad_width():
    from deeplearningrecommendationsystem_b200 import _lib
    import ctypes as C
    lib = _lib.load()
    t = torch.zeros(64, device="cuda")
    f = torch.zeros(8, dtype=torch.uint8, device="cuda")
    P = (C.c_void_p * 1)(t.data_ptr())
    Fl = (C.c_void_p * 1)(f.data_ptr())
    u = _lib.rs_update()
    u.mode, u.width, u.step = _lib.RS_UPD_GRAD, 8, 1
    assert lib.rs_replica_update(P, P, Fl, 64, 1, 0, C.byref(u), None) != 0
    assert b"RS_UPD_SGD or RS_UPD_ADAM" in lib.rs_last_error()
    u.mode, u.width = _lib.RS_UPD_SGD, 6
    assert lib.rs_replica_update(P, P, Fl, 64, 1, 0, C.byref(u), None) != 0


def _batch(rank, step, B, cards):
    g = torch.Generator().manual_seed(900 + 10 * rank + step)
    ids = torch.stack([(torch.rand(B, generator=g) ** 2 * c).long().clamp_(max=c - 1) for c in cards], dim=1)
    return ids, (torch.rand(B, 1, generator=g) < 0.3).float()


def _adam_close(got, want, atol, bound, what):
    """DESIGN.md section 2: Adam divides by sqrt(v), so an element whose summed gradient is at rounding-noise level (a sum
    the single-GPU step associates differently) can land anywhere in a noise-decided range in two fp32 implementations.
    Elements outside rtol 1e-5 / atol must therefore be under 1 % of the tensor and stay within `bound` (w: steps * lr;
    m, v: 1e-5 of the tensor's largest magnitude).  Returns how many such elements there were."""
    bad = ~np.isclose(got, want, rtol=1e-5, atol=atol)
    n = int(bad.sum())
    if n:
        assert n <= 0.01 * got.size, f"{what}: {n} of {got.size} elements beyond tolerance"
        assert np.abs(got - want).max() <= bound, f"{what}: an element differs by more than {bound}"
    return n


def _hybrid_run(world, kind, D, cards, replicate_below, opt_kind, lr, wd, steps=3, B=300):
    from deeplearningrecommendationsystem_b200 import dist as rsdist, ops
    from deeplearningrecommendationsystem_b200.nfield import FieldFFM, FieldFM
    from deeplearningrecommendationsystem_b200.optim import FusedRowOptimizer
    cls = FieldFM if kind == "fm" else FieldFFM
    ref = cls(cards, D, fused=True, seed=4, device="cpu")
    bce = torch.nn.BCELoss()

    def rank_fn(fab):
        m = cls(cards, D, fused=True, seed=4, device="cuda", sharded=True, fabric=fab, replicate_below=replicate_below)
        assert m.hybrid
        m.load_global(ref.weight.data)
        opt = FusedRowOptimizer(m, torch.optim.SGD([m.bias], lr=lr), lr=lr, kind=opt_kind, weight_decay=wd)
        hist = []
        ids, y = _batch(fab.rank, 0, B, cards)
        ids, y = ids.cuda(), y.cuda()                # one batch tensor per rank, stepped on repeatedly (as test_shard_gpu does)
        for s in range(steps):
            w_before = m.weight_small.data.clone()
            opt.zero_grad()
            bce(m(ids), y).backward()
            opt.step()
            hist.append({"w_before": w_before, "gsmall": m.gsmall.clone(), "w": m.weight_small.data.clone(),
                         "m": None if m.adam_m_small is None else m.adam_m_small.clone(),
                         "v": None if m.adam_v_small is None else m.adam_v_small.clone()})
        return {"weight": m.weight.data.clone(), "m": None if m.adam_m is None else m.adam_m.clone(),
                "v": None if m.adam_v is None else m.adam_v.clone(), "hist": hist, "model": m}

    outs = rsdist.ThreadFabric.run(world, rank_fn)
    ops.check_status()
    model0 = outs[0]["model"]
    for r in range(1, world):                   # the replicas must be bit-identical
        assert torch.equal(outs[r]["model"].weight_small.data, model0.weight_small.data)

    # exact check: each step of the replicated rows == the row-update kernel applied to the rank-ordered sum of the ranks'
    # gradient snapshots over the union of the rows the ranks' batches touched
    W = model0.width
    m_prev = torch.zeros(model0.small_total, W, device="cuda")
    v_prev = torch.zeros_like(m_prev)
    touched_ever = set()
    for s in range(steps):
        rows = set()
        for r in range(world):
            ids, _ = _batch(r, 0, B, cards)
            for k, f in enumerate(model0.small_fields):
                rows.update((ids[:, f] + model0.small_offsets_host[k]).tolist())
            touched_ever.update((ids + torch.tensor(model0.offsets_host)).reshape(-1).tolist())
        rows_hit = torch.tensor(sorted(rows), dtype=torch.int64)
        w = outs[0]["hist"][s]["w_before"].clone()
        for r in range(world):
            assert torch.equal(outs[r]["hist"][s]["w_before"], w)
        m_ref, v_ref = m_prev.clone(), v_prev.clone()
        gsum = _rank_sum([outs[r]["hist"][s]["gsmall"].cpu() for r in range(world)])
        _reference_update(ops, w, m_ref, v_ref, rows_hit, gsum, opt_kind, lr, wd, s + 1)
        assert torch.equal(outs[0]["hist"][s]["w"], w), f"step {s}: replicated w differs from the row-update kernel"
        if opt_kind == "adam":
            got_m = torch.cat([outs[r]["hist"][s]["m"] for r in range(world)]).view_as(m_ref)
            got_v = torch.cat([outs[r]["hist"][s]["v"] for r in range(world)]).view_as(v_ref)
            assert torch.equal(got_m, m_ref) and torch.equal(got_v, v_ref), f"step {s}: replicated m / v differ"
            m_prev, v_prev = got_m, got_v

    # the single-GPU step on the concatenated batches
    m = cls(cards, D, fused=True, seed=4, device="cpu").cuda()
    w_init = m.weight.data.clone()
    opt = FusedRowOptimizer(m, torch.optim.SGD([m.bias], lr=lr), lr=lr, kind=opt_kind, weight_decay=wd)
    bs = [_batch(r, 0, B, cards) for r in range(world)]
    ids_all, y_all = torch.cat([b[0] for b in bs]).cuda(), torch.cat([b[1] for b in bs]).cuda()
    for s in range(steps):
        opt.zero_grad()
        bce(m(ids_all), y_all).backward()
        opt.step()
    full = model0.assemble_global([o["weight"] for o in outs])
    noisy = 0
    if opt_kind == "adam":
        noisy = _adam_close(full.cpu().numpy(), m.weight.data.cpu().numpy(), 2e-6, steps * lr * (1 + 1e-6), f"world {world} {kind}: w")
        for name, atol in (("m", 1e-9), ("v", 1e-12)):
            small = torch.cat([getattr(o["model"], f"adam_{name}_small") for o in outs])
            got = model0.assemble_global([o[name] for o in outs], small=small).cpu().numpy()
            want = (m.adam_m if name == "m" else m.adam_v).cpu().numpy()
            noisy += _adam_close(got, want, atol, 1e-5 * np.abs(want).max(), f"world {world} {kind}: {name}")
    else:
        np.testing.assert_allclose(full.cpu().numpy(), m.weight.data.cpu().numpy(), rtol=1e-5, atol=2e-6)
    untouched = torch.ones(model0.total_rows, dtype=torch.bool)
    untouched[torch.tensor(sorted(touched_ever))] = False
    assert untouched.any()
    assert torch.equal(full[untouched.cuda()], w_init[untouched.cuda()]), "a row no step touched moved"
    return noisy


@pytest.mark.parametrize("world", [1, 2, 3, 8])
@pytest.mark.parametrize("kind,D", [("fm", 16), ("ffm", 8), ("ffm", 16)])
@pytest.mark.parametrize("opt_kind", ["adam", "sgd"])
def test_hybrid_lazy_update_equals_single_gpu(world, kind, D, opt_kind):
    """hybrid placement (tables under 100 rows replicated) with Adam or SGD and weight decay, three steps == the
    single-GPU FusedRowOptimizer on the concatenated batch; the replicated rows equal the row-update kernel exactly"""
    lr = ADAM_LR if opt_kind == "adam" else SGD_LR
    noisy = _hybrid_run(world, kind, D, CARDS, 100, opt_kind, lr, WD)
    print(f"[replica-update] world {world} {kind} D={D} {opt_kind}: {noisy} noise-level Adam elements (w, m, v)")


@pytest.mark.parametrize("opt_kind", ["adam", "sgd"])
def test_hybrid_lazy_update_c2_shape(opt_kind):
    """the C2 field layout (cardinalities capped at 2000, tables under 2000 rows replicated) on 4 virtual ranks"""
    lr = ADAM_LR if opt_kind == "adam" else SGD_LR
    for kind in ("ffm", "fm"):
        noisy = _hybrid_run(4, kind, 16, C2_CAPPED, 2000, opt_kind, lr, WD, steps=3, B=700)
        print(f"[replica-update] c2 {kind} {opt_kind}: {noisy} noise-level Adam elements (w, m, v)")


@pytest.mark.parametrize("kind,D", [("fm", 16), ("ffm", 8)])
def test_plain_sgd_keeps_replica_sgd(monkeypatch, kind, D):
    """SGD without weight decay keeps the benchmarked launches: no flags, no lazy update, rs_replica_sgd"""
    ops = _ops()

    def refuse(*a, **k):
        raise AssertionError("plain SGD must not take the lazy replicated update")
    monkeypatch.setattr(ops, "mark_rows", refuse)
    monkeypatch.setattr(ops, "replica_update", refuse)
    _hybrid_run(3, kind, D, CARDS, 100, "sgd", SGD_LR, 0.0)


def test_hybrid_sgd_with_weight_decay_is_graph_capturable():
    """the flag memset and rs_mark_rows capture into a CUDA graph: replays equal eager steps bit for bit"""
    from deeplearningrecommendationsystem_b200 import dist as rsdist
    from deeplearningrecommendationsystem_b200.graph import GraphedTrainStep
    from deeplearningrecommendationsystem_b200.nfield import FieldFFM
    from deeplearningrecommendationsystem_b200.optim import FusedRowOptimizer
    from deeplearningrecommendationsystem_b200.trainer import Trainer
    ms = [FieldFFM(CARDS, 8, seed=2, device="cuda", sharded=True, fabric=rsdist.LocalFabric(), replicate_below=100) for _ in range(2)]
    assert ms[0].hybrid
    ms[1].weight.data.copy_(ms[0].weight.data)
    ms[1].weight_small.data.copy_(ms[0].weight_small.data)
    opts = [FusedRowOptimizer(m, torch.optim.SGD([m.bias], lr=0.1), lr=0.1, weight_decay=WD) for m in ms]
    gs = GraphedTrainStep(ms[0], torch.nn.BCELoss(), opts[0], warmup=1)
    tr = Trainer(ms[1], torch.nn.BCELoss(), opts[1])
    w0 = ms[0].weight_small.data.clone()
    for k in range(5):
        ids, y = _batch(0, k, 256, CARDS)
        ids, y = ids.cuda(), y.cuda()
        gs(ids, rating=y)
        tr.train_loop(ids, train_rating=y)
    torch.cuda.synchronize()
    assert gs.graph is not None
    assert not torch.equal(ms[0].weight_small.data, w0)
    assert torch.equal(ms[0].weight_small.data, ms[1].weight_small.data)
    assert torch.equal(ms[0].weight.data, ms[1].weight.data) and torch.equal(ms[0].bias.data, ms[1].bias.data)


def test_hybrid_adam_two_forwards_raise():
    from deeplearningrecommendationsystem_b200 import dist as rsdist
    from deeplearningrecommendationsystem_b200.nfield import FieldFM
    from deeplearningrecommendationsystem_b200.optim import FusedRowOptimizer

    def rank_fn(fab):
        m = FieldFM(CARDS, 16, seed=4, device="cuda", sharded=True, fabric=fab, replicate_below=100)
        assert m.hybrid
        opt = FusedRowOptimizer(m, None, lr=ADAM_LR, kind="adam", weight_decay=1e-5)
        ids, y = _batch(fab.rank, 0, 64, CARDS)
        ids, y = ids.cuda(), y.cuda()
        opt.zero_grad()
        bce = torch.nn.BCELoss()
        (bce(m(ids), y) + bce(m(ids), y)).backward()
        opt.step()

    with pytest.raises(RuntimeError, match="one forward per optimizer step"):
        rsdist.ThreadFabric.run(2, rank_fn)
