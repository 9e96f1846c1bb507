"""The row-sharded and hybrid train steps of C2 (FM + FFM on the Criteo cardinalities) and C5 (MF on two 100 M-row tables)
at their real table sizes, on N virtual ranks of one GPU (dist.ThreadFabric, as tests/test_shard_gpu.py), each step checked
against a float64 sparse reference of the same step on the concatenated N x B batch.

The sharded step addresses rows through its own arithmetic: request entries packed by shard_post_kernel, the serve kernels'
row offsets into the owner's shard and the requesters' blocks, the direct-field producer of the FFM forward reading the
owners' shards, route_row storing gradient rows into the owners' receive buffers, and the owner's update of its shard.  At
these sizes a shard passes 2^32 floats (N = 2: 16.9 M FFM rows x 416 floats, 1e8 MF rows x 64 floats) or 2^32 bytes
(N = 8 FFM), so an offset truncated to 32 bits would land inside the same allocation, fault nothing and update the wrong
row.  Every rank's batch therefore pins, besides row 0 and the last row of every field, each rank's highest local row and
the first local rows whose float offset reaches 2^31 and 2^32 and whose byte offset reaches 2^32 -- rows other ranks
request as well as the owner's own lookups.

Each step is checked four ways: every rank's predictions and loss, and the bias on every rank; every element of every
touched row, read back from the shard that owns it or from the replicated copy (with Adam also m and v); the replicated
small tables bit-identical on every rank and unchanged where no rank touched them; and bit-identity of the rows the step
must not touch -- a seeded sample of over a million rows of the sharded fields and the 32-bit wrap images of every touched
row relative to its own shard and to the sharded sub-table.

The ranks snapshot the rows they own before the first step and after each step (guard rows as int32, compared on the rank);
the main thread assembles the snapshots and runs sparse_sgd_reference per step.  The ranks take turns on the GPU, so each
case runs the kernels and launch order of the N-GPU step, not its overlap.
"""
import bisect
import gc

import numpy as np
import pytest
import torch

from test_full_scale_gpu import (C2_CARDS, C5_ROWS, D, GUARD_SAMPLE, LR, _field_trainer, assert_rows_match, big_case,  # noqa: F401
                                 guard_sample, make_batch, need_free, sparse_sgd_reference, wrap_images)
from test_replica_update_gpu import _adam_close
from test_segment_update_gpu import B1, B2, EPS, _step64      # betas and eps as the kernels take them (float32)

pytestmark = pytest.mark.gpu
STEPS, WD = 2, 1e-2


# ---------------------------------------------------------------------------------------------- layout, batches, guard rows
def _pins(sub_cards, sub_fields, world, width):
    """(field, id) of the rows every rank's batch pins: for every rank its highest local row and, where its shard has them,
    the first local rows whose float offset reaches 2^31 and 2^32 and whose byte offset reaches 2^32"""
    offs = [sum(sub_cards[:k]) for k in range(len(sub_cards))]
    total = sum(sub_cards)
    firsts = {-(-(1 << 30) // width), -(-(1 << 31) // width), -(-(1 << 32) // width)}
    out = []
    for r in range(world):
        n = (total - r + world - 1) // world
        for local in sorted({n - 1} | {x for x in firsts if x < n}):
            s = local * world + r                                  # row of the sharded sub-table
            k = bisect.bisect_right(offs, s) - 1
            out.append((sub_fields[k], s - offs[k]))
    return out


def _batches(cards, dist, seed, world, nb, pins):
    """make_batch per rank (seed + rank), then every pinned row in every rank's batch (samples 2, 3, ... of its field;
    make_batch's own pins sit at samples 0, 1, nb/3, nb/2 and nb - 1)"""
    out = []
    for r in range(world):
        ids, y = make_batch(cards, dist, seed + r, nb)
        used = {}
        for f, i in pins:
            j = 2 + used.get(f, 0)
            used[f] = used.get(f, 0) + 1
            ids[j, f] = i
        out.append((ids, y))
    return out


class _Layout:
    """Where each distinct row of the global batch lives: the replicated small table (hybrid placement) or the shard of
    rank s % N at local row s // N, s = its row in the row-sharded sub-table; plus the guard rows of every shard."""

    def __init__(self, cards, small, width, world, keys, seed):
        dev = keys.device
        F = len(cards)
        self.small = small
        self.big = [f for f in range(F) if f not in small]
        self.sub_cards = [cards[f] for f in self.big]
        offs = torch.tensor([sum(cards[:k]) for k in range(F)], device=dev)
        small_off = torch.zeros(F, dtype=torch.int64, device=dev)
        sub_off = torch.zeros(F, dtype=torch.int64, device=dev)
        is_small = torch.zeros(F, dtype=torch.bool, device=dev)
        for k, f in enumerate(small):
            small_off[f], is_small[f] = sum(cards[g] for g in small[:k]), True
        for k, f in enumerate(self.big):
            sub_off[f] = sum(self.sub_cards[:k])
        self.uniq, self.inv = torch.unique(keys, return_inverse=True)
        field = torch.searchsorted(offs, self.uniq, right=True) - 1
        local_id = self.uniq - offs[field]
        sm = is_small[field]
        self.small_idx = sm.nonzero().view(-1)                                 # into uniq
        self.small_rows = (small_off[field] + local_id)[self.small_idx]        # into the replicated table
        big_idx = (~sm).nonzero().view(-1)
        sub = (sub_off[field] + local_id)[big_idx]
        self.own_idx = [big_idx[sub % world == r] for r in range(world)]
        self.own_local = [sub[sub % world == r] // world for r in range(world)]
        # guard rows, as rows of the sub-table: a sample over every sharded field and the wrap images of every touched row
        # relative to the sub-table and to its own shard, minus the touched rows
        sub_total = sum(self.sub_cards)
        zero = torch.zeros_like(sub)
        images = [wrap_images(sub, zero, width)]
        for r in range(world):
            loc = self.own_local[r]
            images.append(wrap_images(loc, torch.zeros_like(loc), width) * world + r)
        images = torch.unique(torch.cat(images))
        images = images[~torch.isin(images, sub)]
        assert images.numel() == 0 or int(images.max()) < sub_total
        sample = guard_sample(self.sub_cards, seed, dev)
        sample = sample[~torch.isin(sample, sub)]
        assert sample.numel() >= GUARD_SAMPLE, sample.numel()
        guard = torch.unique(torch.cat([sample, images]))
        self.n_images, self.n_guard, self.n_sample = int(images.numel()), int(guard.numel()), int(sample.numel())
        self.guard_local = [guard[guard % world == r] // world for r in range(world)]

    def assemble(self, per_rank, small=None):
        """(U, W) rows of uniq from every rank's rows of own_local (and the replicated table for the small fields)"""
        out = torch.empty(self.uniq.numel(), per_rank[0].shape[1], dtype=per_rank[0].dtype, device=per_rank[0].device)
        for idx, rows in zip(self.own_idx, per_rank):
            out[idx] = rows
        if self.small:
            out[self.small_idx] = small[self.small_rows]
        return out


# ---------------------------------------------------------------------------------------------- one case
def run_sharded(kind, world, nb, dist, seed, replicate_below, opt_kind="sgd", wd=0.0, expect_direct=None):
    """STEPS steps of Trainer.train_loop on N virtual ranks, one batch per rank; every step checked on its own against
    sparse_sgd_reference on the concatenated batch, started from the rows as the ranks read them before that step."""
    from deeplearningrecommendationsystem_b200 import dist as rsdist, ops
    from deeplearningrecommendationsystem_b200.nfield import FieldFFM, FieldFM, FieldMF
    if kind == "mf":
        cards, width, dim = [C5_ROWS, C5_ROWS], 64, None
        make = lambda **kw: FieldMF(C5_ROWS, C5_ROWS, 64, **kw)          # noqa: E731
    else:
        cards, dim = C2_CARDS, D
        width = D * len(cards) if kind == "ffm" else D
        cls = FieldFFM if kind == "ffm" else FieldFM
        make = lambda **kw: cls(C2_CARDS, D, **kw)                        # noqa: E731
    small = [f for f, c in enumerate(cards) if c < replicate_below] if kind != "mf" else []
    big = [f for f in range(len(cards)) if f not in small]
    pins = _pins([cards[f] for f in big], big, world, width)
    batches = _batches(cards, dist, seed, world, nb, pins)
    offs = torch.tensor([sum(cards[:k]) for k in range(len(cards))], device="cuda")
    L = _Layout(cards, small, width, world, torch.cat([ids + offs for ids, _ in batches]), seed=5)
    y_all = torch.cat([y for _, y in batches])
    adam = opt_kind == "adam"
    torch.cuda.synchronize()

    def rank_fn(fab):
        r = fab.rank
        m = make(fused=True, seed=2, device="cuda", sharded=True, fabric=fab, replicate_below=replicate_below)
        assert m.hybrid == bool(small) and m.big_fields == big and m.weight.shape[0] == fab_rows(r)
        if expect_direct is not None:
            assert bool(m.direct_fields) == expect_direct, m.direct_fields
        tr = _field_trainer(m, opt_kind, wd)
        ids, y = batches[r]
        inputs = (ids[:, 0].contiguous(), ids[:, 1].contiguous()) if kind == "mf" else (ids,)
        loc, gl = L.own_local[r], L.guard_local[r]
        guard0 = m.weight.data[gl].view(torch.int32).clone()
        out = {"rows0": m.weight.data[loc].clone(), "small0": m.weight_small.data.clone() if small else None,
               "bias0": float(m.bias.detach()), "steps": []}
        for _ in range(STEPS):
            tr.train_loop(*inputs, train_rating=y if kind == "mf" else y.view(-1, 1))
            ops.check_status()
            changed = ~(m.weight.data[gl].view(torch.int32) == guard0).all(1)
            st = {"pred": tr.predictions_train.detach().reshape(-1).clone(), "loss": float(tr.train_loss),
                  "bias": float(m.bias.detach()), "rows": m.weight.data[loc].clone(),
                  "changed": int(changed.sum()), "first_changed": int(gl[changed][0]) if bool(changed.any()) else None}
            if small:
                st["small"] = m.weight_small.data.clone()
            if adam:
                st.update(m=m.adam_m[loc].clone(), v=m.adam_v[loc].clone())
                if small:
                    st.update(m_small=m.adam_m_small.clone(), v_small=m.adam_v_small.clone())
            out["steps"].append(st)
        return out

    def fab_rows(r):
        return (sum(cards[f] for f in big) - r + world - 1) // world

    outs = rsdist.ThreadFabric.run(world, rank_fn)
    ops.check_status()
    gc.collect()                  # the ranks' shards and buffers, before the reference allocates
    torch.cuda.empty_cache()
    worst, noisy = [], 0
    prev = {"rows": [o["rows0"] for o in outs], "small": outs[0]["small0"], "bias": outs[0]["bias0"], "m": None, "v": None}
    for s in range(STEPS):
        what = f"{kind} N={world} {dist} step {s + 1}"
        steps = [o["steps"][s] for o in outs]
        for r, st in enumerate(steps):
            assert st["changed"] == 0, (f"{what}: {st['changed']} of {L.guard_local[r].numel()} untouched rows of rank {r}'s shard "
                                        f"changed, first local row {st['first_changed']} ({L.n_images} of the {L.n_guard} guard "
                                        "rows are 32-bit wrap images of touched rows)")
        before = L.assemble(prev["rows"], prev["small"])
        ref = sparse_sgd_reference(kind, before, L.inv, y_all, LR, None if kind == "mf" else prev["bias"], dim=dim)
        # predictions and loss of every rank's slice of the global batch
        p64, y64 = ref["pred"], y_all.double()
        bce = -(y64 * torch.clamp(torch.log(p64), min=-100.0) + (1 - y64) * torch.clamp(torch.log(1 - p64), min=-100.0))
        for r, st in enumerate(steps):
            sl = slice(r * nb, (r + 1) * nb)
            np.testing.assert_allclose(st["pred"].cpu().numpy(), p64[sl].cpu().numpy(), rtol=1e-5, atol=1e-6, err_msg=f"{what} rank {r}")
            np.testing.assert_allclose(st["loss"], float(bce[sl].mean()), rtol=1e-5, err_msg=f"{what} rank {r} loss")
        if kind != "mf":
            assert all(st["bias"] == steps[0]["bias"] for st in steps), f"{what}: the bias differs between ranks"
            np.testing.assert_allclose(steps[0]["bias"], ref["bias"], rtol=1e-5, err_msg=f"{what} bias")
        # the replicated tables: bit-identical on every rank, untouched rows unchanged
        if small:
            s0 = steps[0]["small"]
            for r, st in enumerate(steps[1:], 1):
                assert torch.equal(st["small"].view(torch.int32), s0.view(torch.int32)), f"{what}: replica of rank {r} differs"
            untouched = torch.ones(s0.shape[0], dtype=torch.bool, device=s0.device)
            untouched[L.small_rows] = False
            assert torch.equal(s0[untouched].view(torch.int32), prev["small"][untouched].view(torch.int32)), \
                f"{what}: an untouched row of a replicated table changed"
        after = L.assemble([st["rows"] for st in steps], steps[0].get("small"))
        if not adam:
            worst.append(assert_rows_match(after, ref, LR, what))
        else:
            noisy += _check_adam(L, steps, prev, before, ref, s + 1, what)
            prev["m"] = L.assemble([st["m"] for st in steps], _small_moment(steps, "m_small", L, before))
            prev["v"] = L.assemble([st["v"] for st in steps], _small_moment(steps, "v_small", L, before))
        del before, ref, after
        prev.update(rows=[st["rows"] for st in steps], small=steps[0].get("small"), bias=steps[0]["bias"])
    ops.check_status()
    return {"touched_rows": int(L.uniq.numel()), "guard_rows": L.n_guard, "wrap_images": L.n_images,
            **({"noise_level_adam_elements": noisy} if adam else {"worst_err_over_bound": max(worst)})}


def _small_moment(steps, name, L, like):
    """an Adam moment of the replicated tables: the ranks' small_slice parts, concatenated in rank order"""
    if not L.small:
        return None
    return torch.cat([st[name] for st in steps]).view(-1, like.shape[1])


def _check_adam(L, steps, prev, before, ref, step, what):
    """m and v against their float64 recurrences on the float64 gradient (from zero moments at step 1: _step64), w against
    float64 Adam applied to the kernel's own m and v, each with _adam_close's tolerance.  Returns _adam_close's count of
    noise-level elements (w, m, v)."""
    w0 = before.double()
    if step == 1:
        _, m64, v64 = _step64(w0, ref["grad"], "adam", LR, WD, B1, B2, EPS)
    else:
        gd = ref["grad"] + WD * w0
        m64 = B1 * prev["m"].double() + (1 - B1) * gd
        v64 = B2 * prev["v"].double() + (1 - B2) * gd * gd
    got_m = L.assemble([st["m"] for st in steps], _small_moment(steps, "m_small", L, before)).double()
    got_v = L.assemble([st["v"] for st in steps], _small_moment(steps, "v_small", L, before)).double()
    noisy = _adam_close(got_m.cpu().numpy(), m64.cpu().numpy(), 1e-9, 1e-5 * float(m64.abs().max()), what + " m")
    noisy += _adam_close(got_v.cpu().numpy(), v64.cpu().numpy(), 1e-12, 1e-5 * float(v64.abs().max()), what + " v")
    w64 = w0 - LR / (1 - B1 ** step) * got_m / (got_v.sqrt() / np.sqrt(1 - B2 ** step) + EPS)
    got_w = L.assemble([st["rows"] for st in steps], steps[0].get("small"))
    return noisy + _adam_close(got_w.cpu().numpy(), w64.cpu().numpy(), 2e-6, LR * (1 + 1e-6), what + " w")


# ---------------------------------------------------------------------------------------------- GPU cases
# Device memory each case needs: the table split over the ranks' shards, the ranks' exchange buffers, Jacobian stashes
# and sort workspaces, the snapshots of the touched rows (three per rank), the guard rows as int32, and the float64
# reference over the touched rows.  Peak allocated and wall time of each case on a B200 (1000 W power limit) are in the
# test docstrings.
FFM_GB, FM_GB, MF_GB = 85, 12, 65


@pytest.mark.parametrize("world,nb,dist", [(2, 65536, "uniform"), (2, 65536, "zipf"), (8, 8192, "uniform")])
def test_c2_ffm_hybrid(world, nb, dist, big_case):
    """FieldFFM(C2_CARDS, 16), hybrid placement (tables under 65536 rows replicated; the forward reads the large fields'
    rows from the owners' shards and writes the split stash), SGD lr 0.05.  Peak allocated / wall on a B200: N = 2 uniform
    73.0 GB / 4-6 s (the file's first case: module load included), zipf 69.3 GB / 0.5 s; N = 8 68.3 GB / 0.5 s."""
    from deeplearningrecommendationsystem_b200.nfield import REPLICATE_ROWS
    free = need_free(FFM_GB)
    info = run_sharded("ffm", world, nb, dist, 40 + 10 * world + (dist == "zipf"), REPLICATE_ROWS)
    big_case["info"] = f"ffm hybrid N={world} B={nb} {dist}: {free}, {info}"


@pytest.mark.parametrize("world,nb,direct", [(2, 32768, "1"), (3, 16384, "1"), (2, 32768, "0")])
def test_c2_ffm_all_sharded(world, nb, direct, big_case, monkeypatch):
    """FieldFFM(C2_CARDS, 16), every table row-sharded (replicate_below=0), SGD lr 0.05.  RS_DIRECT=1 (the default): the
    fields of >= 2^20 rows are read from the owners' shards inside the forward kernel; RS_DIRECT=0: every row goes through
    the block fetch (the TMA serve kernel with 1664-byte rows).  N = 3: 33.8 M rows do not divide by 3, so the shards
    differ in length.  B per rank is half the bench's (N = 2) or a quarter (N = 3) because every lookup, not just the
    large fields', goes through the exchange buffers.  Peak allocated / wall on a B200: 71.9 GB / 0.3 s (N = 2, either
    RS_DIRECT), 69.0 GB / 0.3 s (N = 3)."""
    free = need_free(FFM_GB)
    monkeypatch.setenv("RS_DIRECT", direct)
    info = run_sharded("ffm", world, nb, "uniform", 70 + world + 10 * int(direct), 0, expect_direct=direct == "1")
    big_case["info"] = f"ffm all-sharded RS_DIRECT={direct} N={world} B={nb}: {free}, {info}"


@pytest.mark.parametrize("world,nb,dist", [(2, 65536, "uniform"), (2, 65536, "zipf"), (8, 8192, "uniform")])
def test_c2_fm_hybrid(world, nb, dist, big_case):
    """FieldFM(C2_CARDS, 16), hybrid placement (the large fields' rows fetched into a block), SGD lr 0.05.  Peak
    allocated / wall on a B200: 4.0 GB / 0.2 s (N = 2 uniform), 3.9 GB / 0.2 s (zipf), 3.6 GB / 0.2 s (N = 8)."""
    from deeplearningrecommendationsystem_b200.nfield import REPLICATE_ROWS
    free = need_free(FM_GB)
    info = run_sharded("fm", world, nb, dist, 90 + 10 * world + (dist == "zipf"), REPLICATE_ROWS)
    big_case["info"] = f"fm hybrid N={world} B={nb} {dist}: {free}, {info}"


def test_c2_fm_hybrid_adam(big_case):
    """FieldFM(C2_CARDS, 16), hybrid placement, FusedRowOptimizer(kind="adam", lr 0.05, weight_decay=1e-2): lazy Adam by
    the owners on the sharded rows and rs_replica_update on the replicated ones (moments kept by each rank for its
    small_slice); the bias takes SGD.  Peak allocated / wall on a B200: 8.4 GB / 1.6 s."""
    from deeplearningrecommendationsystem_b200.nfield import REPLICATE_ROWS
    free = need_free(FM_GB)
    info = run_sharded("fm", 2, 65536, "uniform", 130, REPLICATE_ROWS, opt_kind="adam", wd=WD)
    big_case["info"] = f"fm hybrid adam N=2 B=65536: {free}, {info}"


@pytest.mark.parametrize("world,nb,dist", [(2, 65536, "uniform"), (2, 65536, "zipf"), (8, 8192, "uniform")])
def test_c5_mf_all_sharded(world, nb, dist, big_case):
    """FieldMF(1e8, 1e8, 64), both tables row-sharded, SGD lr 0.05.  Peak allocated / wall on a B200: 53.0 GB / 0.2 s
    (N = 2 uniform), 52.8 GB / 0.2 s (zipf), 52.6 GB / 0.3 s (N = 8)."""
    free = need_free(MF_GB)
    info = run_sharded("mf", world, nb, dist, 140 + 10 * world + (dist == "zipf"), 0)
    big_case["info"] = f"mf all-sharded N={world} B={nb} {dist}: {free}, {info}"
