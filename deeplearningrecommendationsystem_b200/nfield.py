"""N-field generalisations of the reference's FM / FFM interaction models for the synthetic Criteo-shaped
configs (BASELINE.json configs[1]: 26 sparse fields, D = 16, B = 65536).

The reference modules are hard-wired to the six MovieLens features; these keep the same arithmetic (FM second
order model/deepfm.py:71-77, FFM pairs model/ffm.py:61-82, sigmoid head, BCELoss outside) for F id-fields.  All F
tables live in ONE concatenated (total_rows, W) tensor; ids are int64 (B, F), local to each field.

With ``sharded=True`` (multi-GPU) the concatenated table is ROW-SHARDED over the process group (global row r on rank
r % N) and every step runs the deduplicated ids / rows / row-gradients all-to-alls of ``dist.RowExchange``; the
result equals the single-GPU step on the concatenated global batch (gradients are averaged over ranks).

Two update modes:
  fused=True   (default) the table is not an autograd leaf.  forward launches the fused lookup+interaction kernel
               and keeps the Jacobian rows; backward only records dL/dcross; ``FusedRowOptimizer.step()`` runs the
               sort / segment-reduce / row-update kernels.
  fused=False  the table is a normal dense-gradient nn.Parameter (the reference's semantics, any torch optimizer);
               the gradient is produced by the same deterministic segment-reduce.
"""
import math

import torch
from torch import nn

from . import ops


def _xavier_concat(cards, width, row_dim, device=None, seed=None):
    """xavier_normal_ per field table, as the reference does for each nn.Embedding (model/deepfm.py:34-41).
    Filled slice by slice in place so a 56 GB table never needs a second copy."""
    out = torch.empty(sum(cards), width, dtype=torch.float32, device=device)
    g = None
    if seed is not None:
        g = torch.Generator(device=out.device).manual_seed(seed)
    r0 = 0
    for c in cards:
        out[r0:r0 + c].normal_(0.0, math.sqrt(2.0 / (c + row_dim)), generator=g)
        r0 += c
    return out


REPLICATE_ROWS = 1 << 16   # multi-GPU: fields with fewer rows are REPLICATED on every rank, the others row-sharded (see _FieldModel)
COLD_ROWS = 1 << 16        # stash-free FFM step: fields with at least this many rows are "cold" (see FieldFFM.bind_row_optimizer)
DIRECT_ROWS = 1 << 20      # fields with at least this many rows are read from the peers' shards by the FFM forward itself


def direct_ranges(cardinalities, threshold=DIRECT_ROWS):
    """Global-row ranges of the fields large enough that a batch's lookups into them are (nearly) all distinct: fetching
    those rows into the block first cannot save traffic, so the row-sharded FieldFFM pulls them over NVLink inside its
    forward kernel (dist.DeviceRowExchange(direct=...), rs_ffm_fwd_peer).  At most 8 ranges (the largest fields)."""
    if not threshold:
        return ()
    off, out = 0, []
    for c in cardinalities:
        if c >= threshold:
            out.append((off, off + int(c)))
        off += int(c)
    out.sort(key=lambda r: r[0] - r[1])
    return tuple(sorted(out[:8]))


class _CrossFn(torch.autograd.Function):
    """Routes dL/dcross into the owning module; the table itself is updated by the fused optimizer."""

    @staticmethod
    def forward(ctx, anchor, cross, owner, token):
        ctx.owner, ctx.token = owner, token
        return cross.clone()

    @staticmethod
    def backward(ctx, g):
        ctx.owner._record(ctx.token, g.contiguous())
        return torch.zeros(1, device=g.device), None, None, None


class _DenseGradFn(torch.autograd.Function):
    """Dense-gradient mode: d loss / d table via the deterministic segment-reduce (RS_UPD_GRAD)."""

    @staticmethod
    def forward(ctx, weight, cross, owner, ids, stash):
        ctx.owner = owner
        ctx.save_for_backward(ids, stash)
        ctx.shape = weight.shape
        return cross.clone()

    @staticmethod
    def backward(ctx, g):
        ids, stash = ctx.saved_tensors
        o = ctx.owner
        segs = ops.dedup_sort(ids, o.F, o.offsets_host, o.total_rows, max_width=o.width)
        grad = torch.zeros(ctx.shape, dtype=torch.float32, device=g.device)
        ops.segment_update(segs, ops.RS_UPD_GRAD, o.width, o.F, stash=stash, scale=g.contiguous(), dense_grad=grad)
        return grad, None, None, None, None


class _EmbedFn(torch.autograd.Function):
    """Fused lookup that hands the field embeddings (and optionally their pairwise inner products) to dense layers:
    forward = rs_fields_fwd(concat[, pairs]); backward = rs_fields_bwd -> per-lookup row gradients (B, F, D), recorded
    for the fused row optimizer instead of being scattered into a dense table gradient."""

    @staticmethod
    def forward(ctx, anchor, owner, token, T, ids, want_pairs):
        out = ops.fields_fwd(T, ids.shape[0], ids.device, ids=ids, concat=True, pairs=want_pairs)
        ctx.owner, ctx.token, ctx.T, ctx.want_pairs = owner, token, T, want_pairs
        ctx.save_for_backward(ids)
        if want_pairs:
            return out["concat"], out["pairs"]
        dummy = out["concat"].new_empty(0)
        ctx.mark_non_differentiable(dummy)
        return out["concat"], dummy

    @staticmethod
    def backward(ctx, g_concat, g_pairs):
        (ids,) = ctx.saved_tensors
        dE = ops.fields_bwd(ctx.T, ids.shape[0], ids.device, ids=ids, g_concat=g_concat.contiguous(),
                            g_pairs=g_pairs.contiguous() if ctx.want_pairs else None)
        ctx.owner._record(ctx.token, dE)
        return torch.zeros(1, device=dE.device), None, None, None, None, None


class _FieldModel(nn.Module):
    supports_hybrid = False

    def __init__(self, cardinalities, width, row_dim, fused=True, seed=None, device=None, sharded=False, group=None,
                 fabric=None, exchange=None, direct_threshold=0, replicate_below=None):
        super().__init__()
        self.cards = [int(c) for c in cardinalities]
        self.F, self.width, self.fused = len(self.cards), width, fused
        offs = [0]
        for c in self.cards:
            offs.append(offs[-1] + c)
        self.offsets_host, self.total_rows = offs[:-1], offs[-1]
        self.sharded, self.exchange, self.hybrid, self._hstream = sharded, None, False, None
        if sharded:
            if not fused:
                raise ValueError("sharded tables are updated by the fused row optimizer (fused=True)")
            from . import dist as rsdist
            # Default: the device-side exchange (dist.DeviceRowExchange) -- plan, row fetch and gradient push are this
            # package's kernels over NVLink peer memory, no host sync, CUDA-graph capturable, at every world size.
            # RS_PEER_EXCHANGE=0 selects the NCCL all-to-all formulation (dist.RowExchange, host-synchronised split sizes),
            # which is also what the gloo CPU tests drive.  `exchange` may also be passed in (shared by several models).
            import os
            on_cuda = torch.device(device if device is not None else "cpu").type == "cuda"
            rep = int(os.environ.get("RS_REPLICATE_ROWS", REPLICATE_ROWS)) if replicate_below is None else int(replicate_below)
            small = [f for f, c in enumerate(self.cards) if c < rep]
            big = [f for f, c in enumerate(self.cards) if c >= rep]
            peer_default = os.environ.get("RS_PEER_EXCHANGE", "1") == "1"
            # HYBRID placement (SURVEY.md 8e): small tables are replicated (dense gradient reduced over the ranks by
            # rs_replica_sgd), only the large ones are row-sharded.  Needs the device-side exchange.
            self.hybrid = bool(self.supports_hybrid and small and big and on_cuda and
                               (getattr(exchange, "device_plan", False) if exchange is not None else peer_default))
            if exchange is not None:
                self.exchange = exchange
            elif peer_default:
                direct = direct_ranges(self.cards, direct_threshold) if (os.environ.get("RS_DIRECT", "1") == "1" and not self.hybrid) else ()
                self.exchange = rsdist.DeviceRowExchange(fabric, direct=direct)
            else:
                self.exchange = rsdist.RowExchange(rsdist.cuda_prims(), group)
            if self.hybrid and getattr(self.exchange, "direct", ()):
                raise ValueError("hybrid placement (replicated small tables) takes an exchange without direct ranges")
            self.small_fields, self.big_fields = (small, big) if self.hybrid else ([], list(range(self.F)))
            sh_cards = [self.cards[f] for f in self.big_fields]          # the row-sharded sub-table
            sh_total = sum(sh_cards)
            self.big_cards, self.big_total = sh_cards, sh_total
            self.big_offsets_host = [sum(sh_cards[:k]) for k in range(len(sh_cards))]
            rows = self.exchange.local_rows(sh_total)
            std = math.sqrt(2.0 / (sh_total / len(sh_cards) + row_dim))
            self.shard_ptrs = None
            if getattr(self.exchange, "device_plan", False) and on_cuda:
                # the shard lives in symmetric (peer-mapped) memory, so that kernels of other ranks can read its rows directly
                R = (sh_total + self.exchange.world - 1) // self.exchange.world
                full, self.shard_ptrs = self.exchange.fabric.alloc((R, width), torch.float32, torch.device(device))
                w = full[:rows]
            else:
                w = torch.empty(rows, width, dtype=torch.float32, device=device)
            g = torch.Generator(device=w.device).manual_seed((seed or 0) * 1000 + self.exchange.rank)
            self.weight = nn.Parameter(w.normal_(0.0, std, generator=g), requires_grad=False)
            self.register_buffer("offsets_dev", torch.tensor(self.offsets_host, dtype=torch.int64, device=device), persistent=False)
            if self.hybrid:
                dev, fab = torch.device(device), self.exchange.fabric
                self.small_cards = [self.cards[f] for f in small]
                self.small_total = sum(self.small_cards)
                self.small_offsets_host = [sum(self.small_cards[:k]) for k in range(len(small))]
                ws, self.small_ptrs = fab.alloc((self.small_total, width), torch.float32, dev)
                ws.copy_(_xavier_concat(self.small_cards, width, row_dim, dev, (seed or 0) + 7919))     # same bits on every rank
                self.weight_small = nn.Parameter(ws, requires_grad=False)
                self.gsmall, self.gsmall_ptrs = fab.alloc((self.small_total, width), torch.float32, dev)
                # rows of the small tables this rank's batch touched (lazy update with Adam or weight decay); allocated with
                # the other symmetric buffers so that no step ever allocates collectively
                self.touched_small, self.touched_ptrs = fab.alloc((self.small_total,), torch.uint8, dev)
                self.adam_m_small = self.adam_v_small = None
                self._big_cols_t = torch.tensor(big, dtype=torch.int64, device=dev)
                self._small_cols_t = torch.tensor(small, dtype=torch.int64, device=dev)
                add = [0] * self.F
                for k, f in enumerate(big):
                    add[f] = self.big_offsets_host[k]
                self._mix_add = torch.tensor(add, dtype=torch.int64, device=dev)
                self._big_mask = sum(1 << f for f in big)
                fab.barrier()
        else:
            self.weight = nn.Parameter(_xavier_concat(self.cards, width, row_dim, device, seed), requires_grad=not fused)
        self.bias = nn.Parameter(torch.zeros(1, device=device))
        self._pending, self._anchor, self._token = {}, None, 0
        self.adam_m = self.adam_v = None

    _offset_cache = {}

    def _offsets_key(self):
        """one shared device tensor per (device, offsets): models with equal field layouts share exchange plans"""
        key = (self.weight.device, tuple(self.offsets_host))
        t = _FieldModel._offset_cache.get(key)
        if t is None:
            t = torch.tensor(self.offsets_host, dtype=torch.int64, device=self.weight.device)
            _FieldModel._offset_cache[key] = t
        return t

    def _field_rows(self, table, fields):
        return torch.cat([table[self.offsets_host[f]:self.offsets_host[f] + self.cards[f]] for f in fields])

    def load_global(self, global_weight):
        """sharded mode: take this rank's share of a full (total_rows, W) table -- the rows r % N == rank of the row-sharded
        fields (all of them unless the placement is hybrid) and a full copy of the replicated small fields."""
        from . import dist as rsdist
        gw = global_weight.to(self.weight.device)
        big = self._field_rows(gw, self.big_fields) if self.hybrid else gw
        self.weight.data.copy_(rsdist.shard_rows(big, self.exchange.rank, self.exchange.world))
        if self.hybrid:
            self.weight_small.data.copy_(self._field_rows(gw, self.small_fields))

    def assemble_global(self, shards, small=None):
        """inverse of load_global (tests / verification): list of every rank's weight shard -> the full (total_rows, W) table
        (the replicated fields are taken from this rank's copy, or from `small`, a full (small_total, W) table).  The same
        call assembles Adam's moments: pass every rank's adam_m and, as `small`, the ranks' adam_m_small slices concatenated
        in rank order (see small_slice)."""
        from . import dist as rsdist
        big = rsdist.unshard_rows(list(shards))
        if not self.hybrid:
            return big
        small = self.weight_small.data if small is None else small.reshape(self.small_total, self.width)
        out = torch.empty(self.total_rows, self.width, dtype=big.dtype, device=big.device)
        for k, f in enumerate(self.big_fields):
            out[self.offsets_host[f]:self.offsets_host[f] + self.cards[f]] = big[self.big_offsets_host[k]:self.big_offsets_host[k] + self.cards[f]]
        for k, f in enumerate(self.small_fields):
            out[self.offsets_host[f]:self.offsets_host[f] + self.cards[f]] = \
                small[self.small_offsets_host[k]:self.small_offsets_host[k] + self.cards[f]].to(big.device)
        return out

    @property
    def small_slice(self):
        """hybrid placement: (lo, hi), the elements of the flat replicated table whose update (and Adam moments,
        adam_m_small / adam_v_small) this rank owns"""
        return ops.replica_slice(self.small_total * self.width, self.exchange.world, self.exchange.rank)

    def tables(self):
        return ops.tables_from_concat(self.weight.data, self.offsets_host, self.cards)

    # --- fused-mode bookkeeping
    def _record(self, token, g):
        if token in self._pending:
            self._pending[token]["g"] = g

    def clear_pending(self):
        self._pending.clear()

    def _row_update(self, opt, segs, F, tag="", **src):
        """Apply the optimizer to the rows of self.weight named by `segs` (gradient source in **src)."""
        if opt.kind == "sgd":
            ops.segment_update(segs, ops.RS_UPD_SGD, self.width, F, table=self.weight.data, lr=opt.lr, wd=opt.weight_decay, tag=tag, **src)
        else:
            if self.adam_m is None:
                self.adam_m = torch.zeros_like(self.weight.data)
                self.adam_v = torch.zeros_like(self.weight.data)
            ops.segment_update(segs, ops.RS_UPD_ADAM, self.width, F, table=self.weight.data, m=self.adam_m, v=self.adam_v,
                               lr=opt.lr, wd=opt.weight_decay, betas=opt.betas, eps=opt.eps, step=opt.step_count, tag=tag, **src)

    def _merged_record(self, recs):
        """The pending records of several forwards as one record over their concatenated batches, so that Adam and weight
        decay step once on the summed gradient (see FusedRowOptimizer).  Stash + per-sample scale are concatenated as they
        are when every record has them; otherwise the stashed rows are multiplied out into per-lookup gradient rows (the
        same fp32 product the update kernels form)."""
        ids = torch.cat([r["ids"] for r in recs])
        if all(r.get("stash") is not None for r in recs):
            return {"ids": ids, "stash": torch.cat([r["stash"] for r in recs]), "g": torch.cat([r["g"] for r in recs])}
        dense = [r["g"].reshape(r["ids"].shape[0], -1, self.width) if r.get("stash") is None else
                 r["stash"].reshape(r["ids"].shape[0], -1, self.width) * r["g"].reshape(-1, 1, 1) for r in recs]
        return {"ids": ids, "stash": None, "g": torch.cat(dense)}

    def apply_pending(self, opt):
        recs = [rec for rec in self._pending.values() if "g" in rec]
        if len(recs) > 1 and (opt.kind != "sgd" or opt.weight_decay != 0.0):
            # several forwards before one step: Adam's moments and the decay term must advance once, on the summed gradient
            if self.sharded:
                raise RuntimeError("a row-sharded table takes one forward per optimizer step with Adam or weight_decay != 0 "
                                   f"({len(recs)} forwards are pending)")
            if any(r.get("recompute") for r in recs):
                raise RuntimeError("a forward without a Jacobian stash cannot be merged with another one before a step with "
                                   "weight_decay != 0; run with RS_FFM_RECOMPUTE=0")
            recs = [self._merged_record(recs)]
        for rec in recs:
            src = {"dense": rec["g"]} if rec.get("stash") is None else {"stash": rec["stash"], "scale": rec["g"]}
            if not self.sharded:
                segs = ops.dedup_sort(rec["ids"], self.F, self.offsets_host, self.total_rows, max_width=self.width)
                if rec.get("recompute"):      # FieldFFM without a Jacobian stash: gradient rows rebuilt from the table itself
                    if opt.kind != "sgd":
                        raise RuntimeError("this forward ran without a Jacobian stash (row optimizer bound as SGD); step it with that optimizer")
                    ops.ffm_bwd_update(self.tables(), rec["ids"], self.D, segs, rec["g"], self.weight.data, opt.lr, opt.weight_decay,
                                       cold_mask=self.cold_mask, cold_stash=rec["stash"])
                    continue
                self._row_update(opt, segs, self.F, **src)
                continue
            if rec.get("hybrid"):
                self._apply_hybrid(opt, rec)
                continue
            # row-sharded: reduce the batch's gradients per fetched row, send them to the owners, update there
            plan, ex = rec["plan"], self.exchange
            if plan.segs is not None:      # the plan already sorted these lookups by row: no second sort
                segs = ops.block_segments(plan.segs, plan.n_uniq, self.width)
            else:
                segs = ops.dedup_sort(plan.local_ids, 1, None, plan.n_uniq, max_width=self.width)   # memoised per plan
            if "scale" in src:
                src["scale"] = src["scale"] * (1.0 / ex.world)          # gradients are averaged over the ranks
            else:
                src["dense"] = src["dense"] * (1.0 / ex.world)
            if getattr(ex, "device_plan", False):
                # segment-reduce fused with the push: every reduced row is stored straight into its owner's buffer over
                # NVLink (device-resident routes); after the barrier the owner runs the same sort / segment-reduce /
                # update kernels over what it received (the fill level of that buffer is a device scalar: n_valid)
                routes, ent = ex.grad_routes(plan, self.weight.data, rec["g"].device)
                ops.segment_update(segs, ops.RS_UPD_GRAD, self.width, self.F, grad_routes=routes, tag="/push", **src)
                recv = ex.finish_push(plan, ent)
                osegs = ex.owner_segments(plan, self.weight.shape[0], self.width)
                self._row_update(opt, osegs, 1, tag="/owner", dense=recv)
                continue
            # NCCL formulation: every fetched row has at least one lookup in this batch, so RS_UPD_GRAD writes every row
            block_grad = torch.empty(plan.n_uniq, self.width, dtype=torch.float32, device=rec["g"].device)
            ops.segment_update(segs, ops.RS_UPD_GRAD, self.width, self.F, dense_grad=block_grad, **src)
            recv = ex.push_grads(plan, block_grad)
            if recv.shape[0]:
                osegs = ops.dedup_sort(plan.recv_local, 1, None, self.weight.shape[0], max_width=self.width)
                self._row_update(opt, osegs, 1, dense=recv)
        self._pending.clear()

    # ---- hybrid placement: replicated small tables + row-sharded large ones
    def _hybrid_tables(self, block):
        """rs_tables of the F fields: small fields -> this rank's replica, large fields -> `block` (rows fetched by the
        exchange; None when the forward kernel reads them from the owners' shards itself)."""
        T = ops._lib.rs_tables()
        T.num_fields, T.width = self.F, self.width
        small_base = self.weight_small.data_ptr()
        for k, f in enumerate(self.small_fields):
            T.base[f] = small_base + self.small_offsets_host[k] * self.width * 4
            T.rows[f] = self.cards[f]
        for f in self.big_fields:
            T.base[f] = block.data_ptr() if block is not None else self.weight.data_ptr()
            T.rows[f] = block.shape[0] if block is not None else 1
        return T

    def _hybrid_forward(self, ids, train):
        ex = self.exchange
        ids_big = ex.derived(ids, "big", lambda: ids[:, self._big_cols_t].contiguous())
        rec = {"hybrid": True}
        plan = None
        if train or not self.hybrid_direct:
            # the plan (sort of the large-field lookups, request lists to the owners) is only needed before the forward if
            # rows have to be fetched; otherwise it runs on a side stream under the forward kernel
            plan = ex.plan_for(ids_big, self.big_offsets_host, self.big_total, on_side=self.hybrid_direct,
                               prefetch_rows=self.weight.shape[0] if train else None, wait=not self.hybrid_direct)
        if train:
            ids_small = ex.derived(ids, "small", lambda: ids[:, self._small_cols_t].contiguous())
            ops.prefetch_dedup(ids_small, len(self.small_fields), self.small_offsets_host, self.small_total)
            rec.update(plan=plan, ids_small=ids_small)
        cross, st_small, st_big = self._hybrid_interact(ids, plan, train)
        rec.update(stash_small=st_small, stash_big=st_big)
        return cross, rec

    def _apply_hybrid(self, opt, rec):
        # plain SGD without decay moves an untouched row by lr * 0: every element is stepped (rs_replica_sgd).  Otherwise the
        # update is lazy, as on one GPU: each rank flags the rows its batch touched and only flagged rows step.
        lazy = opt.kind != "sgd" or opt.weight_decay != 0.0
        ex, W = self.exchange, self.width
        plan = rec["plan"]
        ex.wait_plan(plan)                       # (before this step's first barrier on this stream)
        g = rec["g"] * (1.0 / ex.world)          # gradients are averaged over the ranks
        Fs, Fb = len(self.small_fields), len(self.big_fields)
        # The two reductions run side by side: the replicated tables' (HBM-bound, local) on a side stream, the sharded
        # tables' (bound by the NVLink stores to the owners) on this one; each streaming kernel takes half of every SM.
        cur = torch.cuda.current_stream()
        if self._hstream is None:
            self._hstream = torch.cuda.Stream(device=g.device)
        self._hstream.wait_stream(cur)
        with torch.cuda.stream(self._hstream):
            # replicated tables: this rank's batch reduced into its dense gradient (symmetric memory)
            segs_s = ops.dedup_sort(rec["ids_small"], Fs, self.small_offsets_host, self.small_total, max_width=W)
            self.gsmall.zero_()
            ops.segment_update(segs_s, ops.RS_UPD_GRAD, W, Fs, stash=rec["stash_small"], scale=g, dense_grad=self.gsmall, tag="/small",
                               half_sm=True)
            if lazy:
                # peers read these flags only after finish_push's barrier, and the barrier that ends the step orders those
                # reads before this zeroing in the next step (the discipline gsmall follows)
                self.touched_small.zero_()
                ops.mark_rows(segs_s, self.touched_small, self.small_total)
            small_done = torch.cuda.Event()
            small_done.record()
        # row-sharded tables: reduce per distinct row, store straight into the owners' buffers
        segs_b = ops.block_segments(plan.segs, plan.n_uniq, W)
        routes, ent = ex.grad_routes(plan, self.weight.data, g.device)
        ops.segment_update(segs_b, ops.RS_UPD_GRAD, W, Fb, grad_routes=routes, stash=rec["stash_big"], scale=g, tag="/push", half_sm=True)
        cur.wait_event(small_done)
        recv = ex.finish_push(plan, ent)         # barrier: pushed rows have landed, every rank's dense gradient is complete
        if not lazy:
            ops.replica_sgd(self.small_ptrs, self.gsmall_ptrs, self.small_total * W, ex.world, ex.rank, opt.lr)
        else:
            if opt.kind == "adam" and self.adam_m_small is None:
                lo, hi = self.small_slice
                self.adam_m_small = torch.zeros(hi - lo, dtype=torch.float32, device=g.device)
                self.adam_v_small = torch.zeros(hi - lo, dtype=torch.float32, device=g.device)
            ops.replica_update(self.small_ptrs, self.gsmall_ptrs, self.touched_ptrs, self.small_total * W, W, ex.world, ex.rank,
                               opt.kind, opt.lr, opt.weight_decay, m=self.adam_m_small, v=self.adam_v_small, betas=opt.betas,
                               eps=opt.eps, step=opt.step_count)
        osegs = ex.owner_segments(plan, self.weight.shape[0], W)
        self._row_update(opt, osegs, 1, tag="/owner", dense=recv)
        from .dist import _phase
        with _phase("exchange_barrier"):
            ex.fabric.barrier()                  # replicas rewritten and gradients read before anyone's next step

    def _plan(self, ids, train):
        ex = self.exchange
        if getattr(ex, "device_plan", False):
            plan = ex.plan_for(ids, self.offsets_host, self.total_rows)
            if train:      # the owner-side sort of the requested rows depends only on the plan: overlap it with fetch + forward
                ex.prefetch_owner_segments(plan, self.weight.shape[0])
            return plan
        plan = ex.plan_for(ids, self._offsets_key(), self.total_rows)
        if train and plan.recv_local.numel():
            ops.prefetch_dedup(plan.recv_local, 1, None, self.weight.shape[0])
        return plan

    def _interact(self, T, ids, want_stash):
        raise NotImplementedError

    def embed(self, ids, want_pairs=False):
        """(B, F*D) concat of the field embeddings [and (B, P) inner products], differentiable for the layers above;
        the table update goes through the fused row optimizer (fused=True only)."""
        if not self.fused:
            raise NotImplementedError("embed() is implemented for fused tables")
        if ids.dim() != 2 or ids.shape[1] != self.F:
            raise ValueError(f"ids must be (B, {self.F})")
        rec = {}
        if self.sharded:
            plan = self._plan(ids, torch.is_grad_enabled())
            block = self.exchange.fetch(plan, self.weight.data)
            ids, T, rec = plan.local_ids.view(ids.shape), ops.make_tables([block] * self.F), {"plan": plan, "block": block}
        else:
            T = self.tables()
        if not torch.is_grad_enabled():
            out = ops.fields_fwd(T, ids.shape[0], ids.device, ids=ids, concat=True, pairs=want_pairs)
            return out["concat"], out.get("pairs")
        if self._anchor is None or self._anchor.device != ids.device:
            self._anchor = torch.zeros(1, device=ids.device, requires_grad=True)
        self._token += 1
        self._pending[self._token] = {"ids": ids, "stash": None, **rec}
        concat, pairs = _EmbedFn.apply(self._anchor, self, self._token, T, ids, want_pairs)
        return concat, (pairs if want_pairs else None)

    def logit(self, ids, add_bias=True):
        if ids.dim() != 2 or ids.shape[1] != self.F:
            raise ValueError(f"ids must be (B, {self.F})")
        train = torch.is_grad_enabled()
        rec = {}
        if self.sharded and self.hybrid:
            cross, rec = self._hybrid_forward(ids, train and self.fused)
            stash = rec.get("stash_small")
        elif self.sharded:
            plan = self._plan(ids, train and self.fused)
            direct = bool(getattr(self, "direct_fields", None))
            if direct:
                block = self.exchange.fetch(plan, self.weight.data, skip_direct=True)
            else:
                block = self.exchange.fetch(plan, self.weight.data)
            orig, ids = ids, plan.local_ids.view(ids.shape)
            cross, stash = self._interact(ops.make_tables([block] * self.F), ids, want_stash=train, **({"orig_ids": orig} if direct else {}))
            rec = {"plan": plan}
        else:
            if train and self.fused:      # the sort depends only on the ids: overlap it with the forward kernels
                ops.prefetch_dedup(ids, self.F, self.offsets_host, self.total_rows)
            cross, stash = self._interact(self.tables(), ids, want_stash=train)
        if train and self.fused:
            if self._anchor is None or self._anchor.device != ids.device:
                self._anchor = torch.zeros(1, device=ids.device, requires_grad=True)
            self._token += 1
            if getattr(self, "_stash_is_cold_slices", False):
                rec = {**rec, "recompute": True}
            self._pending[self._token] = {"ids": ids, "stash": stash, **rec}
            cross = _CrossFn.apply(self._anchor, cross, self, self._token)
        elif train:
            cross = _DenseGradFn.apply(self.weight, cross, self, ids, stash)
        return cross + self.bias if (self.use_bias and add_bias) else cross

    use_bias = True

    def forward(self, ids):
        return torch.sigmoid(self.logit(ids)).unsqueeze(1)

    def train_logit(self, ids):
        """(cross (B,), bias parameter | None, shape of forward()'s output) with logit = cross + bias -- lets the Trainer fuse
        the bias add, sigmoid, BCELoss, their backward and the bias-gradient sum into one kernel pair"""
        return self.logit(ids, add_bias=False), (self.bias if self.use_bias else None), (ids.shape[0], 1)


class FieldFM(_FieldModel):
    """sigmoid(b + 0.5 * sum_d[(sum_f e_f)^2 - sum_f e_f^2]) over F id-fields, D-dim rows."""

    def __init__(self, cardinalities, embedding_dim, fused=True, seed=None, device=None, sharded=False, group=None, **kw):
        super().__init__(cardinalities, embedding_dim, embedding_dim, fused, seed, device, sharded, group, **kw)

    supports_hybrid = True
    hybrid_direct = False        # the large-field rows are fetched into a block before the forward

    def _interact(self, T, ids, want_stash):
        out = ops.fields_fwd(T, ids.shape[0], ids.device, ids=ids, cross=True, stash=want_stash)
        return out["cross"], out.get("stash")

    def _hybrid_interact(self, ids, plan, want_stash):
        block = self.exchange.fetch(plan, self.weight.data)
        mix = ids.clone()
        mix[:, self._big_cols_t] = plan.local_ids.view(ids.shape[0], len(self.big_fields))
        out = ops.fields_fwd(self._hybrid_tables(block), ids.shape[0], ids.device, ids=mix, cross=True, stash=want_stash)
        if not want_stash:
            return out["cross"], None, None
        st = out["stash"]                                   # (B, F, D): 64-byte rows, split by a gather
        return out["cross"], st[:, self._small_cols_t].contiguous(), st[:, self._big_cols_t].contiguous()


class FieldFFM(_FieldModel):
    """sigmoid(b + sum_{i<j} <v_{i,j}, v_{j,i}>): feature i's table row is (F, D), slot j aimed at field j."""

    def __init__(self, cardinalities, num_vector, fused=True, seed=None, device=None, sharded=False, group=None,
                 direct_threshold=DIRECT_ROWS, **kw):
        F = len(cardinalities)
        super().__init__(cardinalities, F * num_vector, num_vector, fused, seed, device, sharded, group,
                         direct_threshold=direct_threshold, **kw)
        self.D = num_vector
        # fields whose whole row range is one of the exchange's direct ranges: the forward kernel reads their rows from the
        # owners' shards itself (see direct_ranges); needs the shard in symmetric memory
        self.direct_fields = []
        ranges = set(getattr(self.exchange, "direct", ()) or ()) if self.sharded and self.shard_ptrs is not None else set()
        for f, (o, c) in enumerate(zip(self.offsets_host, self.cards)):
            if (o, o + c) in ranges:
                self.direct_fields.append(f)
        if self.direct_fields:
            dev = self.weight.device
            self._direct_cols = torch.tensor(self.direct_fields, dtype=torch.int64, device=dev)
            self._direct_offs = torch.tensor([self.offsets_host[f] for f in self.direct_fields], dtype=torch.int64, device=dev)
            self._direct_mask = sum(1 << f for f in self.direct_fields)

    supports_hybrid = True
    hybrid_direct = True         # the forward kernel reads the large-field rows from the owners' shards itself

    def _hybrid_interact(self, ids, plan, want_stash):
        mix = ids + self._mix_add                           # large fields: global row inside the sharded sub-table
        peer = (self.exchange.world, self._big_mask, self.shard_ptrs, self.big_total)
        if not want_stash:
            cross, _ = ops.ffm_fwd(self._hybrid_tables(None), mix, self.D, want_stash=False, peer=peer)
            return cross, None, None
        return ops.ffm_fwd(self._hybrid_tables(None), mix, self.D, want_stash=True, peer=peer, split_mask=self._big_mask)

    def bind_row_optimizer(self, opt):
        """Called by FusedRowOptimizer.  RS_FFM_RECOMPUTE=1 (opt-in; plain SGD, unsharded table): the training forward
        writes only a cold-slice stash and the step rebuilds the gradient rows from the table (ops.ffm_fwd_train /
        ops.ffm_bwd_update), bit-identical to the default.  It moves about half the DRAM bytes of the full-stash step but
        is SLOWER on B200 (4.5 vs 2.2 ms per C2 step): its 64-byte slice gathers run at ~27 G accesses/s, while the
        full-stash kernels stream 1664-byte rows through TMA at 5 TB/s (DESIGN.md section 4, profiles/r2_ffm_stash_free.md)."""
        import os
        self._recompute = (opt.kind == "sgd" and self.fused and not self.sharded and self.width // 4 <= 256
                           and os.environ.get("RS_FFM_RECOMPUTE", "0") == "1")
        # "cold" fields: tables too large to stay in L2.  Their once-looked-up rows are updated in place, and slices that
        # live in their rows travel through the cold-slice stash instead of being gathered at random from a many-GB table.
        self.cold_mask = sum(1 << f for f, c in enumerate(self.cards) if c >= COLD_ROWS)

    def _interact(self, T, ids, want_stash, orig_ids=None):
        self._stash_is_cold_slices = False
        if want_stash and getattr(self, "_recompute", False) and self.fused and not self._pending:
            # (a second forward before the step keeps its full stash: its gradients must not see the first one's update)
            self._stash_is_cold_slices = True
            return ops.ffm_fwd_train(T, ids, self.D, self.cold_mask)
        if orig_ids is not None and self.direct_fields:
            # block rows for the fetched fields, GLOBAL rows for the direct ones
            mix = ids.clone()
            mix[:, self._direct_cols] = orig_ids[:, self._direct_cols] + self._direct_offs
            return ops.ffm_fwd(T, mix, self.D, want_stash=want_stash,
                               peer=(self.exchange.world, self._direct_mask, self.shard_ptrs, self.total_rows))
        return ops.ffm_fwd(T, ids, self.D, want_stash=want_stash)


class FieldMF(_FieldModel):
    """sigmoid(<U[u], V[i]>) with the user and item tables in one concatenated (optionally row-sharded) buffer --
    the large-table form of reference model/mf.py:11-26 (same forward signature and 1-D output) for the synthetic
    100 M-row configs.  d dot / d U[u] = V[i] is exactly the FM Jacobian S - e for two fields, so the fused lookup
    kernel's stash and the segment-reduce/update path are shared with FieldFM."""

    use_bias = False

    def __init__(self, num_users, num_items, embedding_size, fused=True, seed=None, device=None, sharded=False, group=None, **kw):
        super().__init__([num_users, num_items], embedding_size, embedding_size, fused, seed, device, sharded, group, **kw)
        self.bias.requires_grad_(False)

    def _interact(self, T, ids, want_stash):
        out = ops.fields_fwd(T, ids.shape[0], ids.device, ids=ids, dot2=True, stash=want_stash)
        return out["dot2"], out.get("stash")

    def forward(self, user_indices, item_indices):
        ids = torch.stack([user_indices, item_indices], dim=1)
        return torch.sigmoid(self.logit(ids))                       # (B,)

    def train_logit(self, user_indices, item_indices):
        ids = torch.stack([user_indices, item_indices], dim=1)
        return self.logit(ids, add_bias=False), None, (ids.shape[0],)


class _EmbedModel(_FieldModel):
    """models that use the table through embed() and put dense layers on top: forward() is not sigmoid(logit())"""
    train_logit = None


class FieldPNN(_EmbedModel):
    """Inner-product PNN over F id-fields (reference model/pnn.py:55-77,111-131 generalised from six features):
    lz = Linear(F*D, H0)(concat), lp = Linear(F(F-1)/2, H0)(inner products), ReLU tower, Linear(H[-1], 1), sigmoid."""

    use_bias = False

    def __init__(self, cardinalities, embed_dim, hidden_units, fused=True, seed=None, device=None, sharded=False, group=None, **kw):
        super().__init__(cardinalities, embed_dim, embed_dim, fused, seed, device, sharded, group, **kw)
        F = self.F
        self.bias.requires_grad_(False)
        self.linear1 = nn.Linear(F * embed_dim, hidden_units[0], device=device)
        self.linear2 = nn.Linear(F * (F - 1) // 2, hidden_units[0], device=device)
        self.dnn_network = nn.ModuleList([nn.Linear(a, b, device=device) for a, b in zip(hidden_units[:-1], hidden_units[1:])])
        self.output = nn.Linear(hidden_units[-1], 1, device=device)

    def forward(self, ids):
        concat, pairs = self.embed(ids, want_pairs=True)
        h = self.linear1(concat) + self.linear2(pairs)
        for layer in self.dnn_network:
            h = torch.relu(layer(h))
        return torch.sigmoid(self.output(h)).view(-1, 1)


class FieldAFM(_EmbedModel):
    """Attentional pooling over the F(F-1)/2 pairwise products of F id-fields (reference model/afm.py:55-66):
    sigmoid(Linear(D,1)(sum_p softmax_p(h.relu(P_p W + b)) P_p))."""

    use_bias = False

    def __init__(self, cardinalities, embed_dim, attention_dim, fused=True, seed=None, device=None, sharded=False, group=None, **kw):
        super().__init__(cardinalities, embed_dim, embed_dim, fused, seed, device, sharded, group, **kw)
        self.bias.requires_grad_(False)
        g = torch.Generator(device="cpu").manual_seed(seed or 0)
        self.attention_W = nn.Parameter((torch.randn(embed_dim, attention_dim, generator=g) * 0.1).to(device))
        self.attention_b = nn.Parameter(torch.zeros(attention_dim, device=device))
        self.attention_h = nn.Parameter((torch.randn(attention_dim, 1, generator=g) * 0.1).to(device))
        self.output_layer = nn.Linear(embed_dim, 1, device=device)

    def forward(self, ids):
        from . import attention
        concat, _ = self.embed(ids)
        pooled = attention.afm_pool(concat.view(ids.shape[0], self.F, self.width), self.attention_W, self.attention_b, self.attention_h)
        return torch.sigmoid(self.output_layer(pooled))


class _PairTable(_EmbedModel):
    """user + item tables of one embedding width in one concatenated (optionally row-sharded) buffer; only embed() is used"""
    use_bias = False

    def __init__(self, num_users, num_items, width, **kw):
        super().__init__([num_users, num_items], width, width, **kw)
        self.bias.requires_grad_(False)


class FieldNeuralCF(nn.Module):
    """NeuralCF (reference model/neuralcf.py:7-59: GMF Hadamard * MLP tower on [u_mlp, i_mlp], Linear(layers[-1], mf_dim),
    Linear(2 mf_dim, 1), sigmoid) for the synthetic 100 M-row configs (BASELINE.json configs[4]): the four embedding tables
    live in two concatenated buffers (GMF user+item, MLP user+item), updated by the fused row optimizer and -- with
    ``sharded=True`` -- row-sharded over the ranks with ONE exchange plan per batch shared by both buffers (same ids, same
    row layout).  Same forward signature and (B, 1) output as the reference module."""

    def __init__(self, num_user, num_item, mf_dim, layers, fused=True, seed=None, device=None, sharded=False, group=None,
                 fabric=None, exchange=None):
        super().__init__()
        if sharded and exchange is None:
            from . import dist as rsdist
            import os
            if os.environ.get("RS_PEER_EXCHANGE", "1") == "1":
                exchange = rsdist.DeviceRowExchange(fabric)
        kw = dict(fused=fused, device=device, sharded=sharded, group=group, exchange=exchange)
        self.gmf = _PairTable(num_user, num_item, mf_dim, seed=seed, **kw)
        self.mlp = _PairTable(num_user, num_item, int(layers[0] / 2), seed=None if seed is None else seed + 1, **kw)
        self.mf_dim = mf_dim
        self.dnn_network = nn.ModuleList([nn.Linear(a, b, device=device) for a, b in zip(layers[:-1], layers[1:])])
        self.linear = nn.Linear(layers[-1], mf_dim, device=device)
        self.linear2 = nn.Linear(2 * mf_dim, 1, device=device)

    def forward(self, user_indices, item_indices):
        ids = torch.stack([user_indices, item_indices], dim=1)
        g, _ = self.gmf.embed(ids)                               # (B, 2 mf_dim) = [U_g[u] | V_g[i]]
        gmf = g[:, :self.mf_dim] * g[:, self.mf_dim:]
        x, _ = self.mlp.embed(ids)                               # (B, layers[0]) = cat[U_m[u], V_m[i]]
        for layer in self.dnn_network:
            x = torch.relu(layer(x))
        return torch.sigmoid(self.linear2(torch.cat([gmf, self.linear(x)], dim=1)))
