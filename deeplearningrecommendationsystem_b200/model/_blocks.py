"""autograd building blocks shared by the drop-in modules.

Every Function's forward and backward is one or two calls into the C ABI (ops.*); torch.autograd only carries
the tensors between them.  Embedding-table gradients are produced by the deterministic sort / segment-reduce
(rs_dedup_sort + rs_segment_update in RS_UPD_GRAD mode) as ordinary dense ``.grad`` tensors, so the reference's
``optim.Adam(model.parameters(), lr, weight_decay=1e-5)`` (scripts/deepfm.py:55) runs unchanged on top.
"""
import torch

from .. import ops

# x (B,45) column layout, data/reader.py:98-101: [uid, iid, age, gender(2), occupation(21), genre(19)]
COL_USER, COL_ITEM = 0, 1
AGE, GENDER, OCC, GENRE = (2, 1), (3, 2), (5, 21), (26, 19)
KIND_ID, KIND_BAG, KIND_SCALAR = 0, 1, 2


def table_grads(ids, dE, rows):
    """Dense gradients of F tables from per-lookup row gradients.

    ids (N, F) int64, dE (N, F, W) fp32, rows[f] = number of rows of table f.  One stable sort over all F fields
    (keys = row offset of the field + id), one fixed-order segment-reduce; the F gradients are views of one buffer.
    """
    F, W = len(rows), dE.shape[-1]
    offs, total = [], 0
    for r in rows:
        offs.append(total)
        total += r
    ids = ids.reshape(-1, F)
    buf = torch.zeros(total, W, dtype=torch.float32, device=dE.device)
    if ids.numel() == 0:
        return [buf[o:o + r] for o, r in zip(offs, rows)]
    segs = ops.dedup_sort(ids, F, offs, total, max_width=W)
    ops.segment_update(segs, ops.RS_UPD_GRAD, W, F, dense=dE.reshape(-1, W), dense_grad=buf)
    return [buf[o:o + r] for o, r in zip(offs, rows)]


class EmbeddingLookup(torch.autograd.Function):
    """weight[ids] for one table -- nn.Embedding.forward / embedding_dense_backward
    (reference model/mf.py:24-25, model/din.py:35-36; backward implicit at trainer/trainer.py:38)."""

    @staticmethod
    def forward(ctx, weight, ids):
        ctx.save_for_backward(ids)
        ctx.rows = weight.shape[0]
        out = ops.gather_rows(ops.make_tables([weight.detach()]), ids.reshape(-1, 1))
        return out.view(*ids.shape, weight.shape[1])

    @staticmethod
    def backward(ctx, g):
        (ids,) = ctx.saved_tensors
        (gw,) = table_grads(ids.reshape(-1, 1), g.contiguous().view(-1, 1, g.shape[-1]), [ctx.rows])
        return gw, None


def lookup(weight, ids):
    sink = getattr(weight, "_rs_sink", None)
    if sink is not None and torch.is_grad_enabled():
        return _FusedLookup.apply(sink.anchor(weight.device), weight, ids)
    return EmbeddingLookup.apply(weight, ids)


# --------------------------------------------------------------------------------------------------------------------
# Opt-in FUSED SPARSE mode for the id-indexed drop-in modules (DIN, DIEN, MatrixFactorization, NeuralCF).
# Reference semantics (nn.Embedding + a dense optimizer, model/din.py:35-36 + trainer/trainer.py:38-39) cost a table-sized
# zero-fill, a table-sized gradient and a full-table optimizer sweep every step -- proportional to the ROW COUNT, not to the
# batch.  After ``model.fuse_embedding_updates()`` the tables stop being autograd leaves: backward hands the per-lookup row
# gradients to a RowSink and ``FusedRowOptimizer.step()`` runs rs_dedup_sort + rs_segment_update (sort / segment-reduce
# fused with the SGD or lazy-Adam row update) on the touched rows only.  SGD without weight decay is exactly the
# reference's update (untouched rows have zero gradient); Adam / weight decay become row-wise (lazy) -- see optim.py.
class RowSink:
    def __init__(self):
        self.groups, self.pending, self._anchor = [], [], None

    def anchor(self, device):
        if self._anchor is None or self._anchor.device != device:
            self._anchor = torch.zeros(1, device=device, requires_grad=True)
        return self._anchor

    def add_group(self, embeddings):
        """Tables of equal width that are looked up together (MF user + item) move into ONE concatenated buffer (each
        nn.Embedding.weight becomes a view of it, state_dict keys and shapes unchanged), so one sort covers them."""
        ws = [e.weight for e in embeddings]
        W, dev = ws[0].shape[1], ws[0].device
        if any(w.shape[1] != W or w.device != dev for w in ws) or dev.type != "cuda":
            raise ValueError("fuse_embedding_updates: move the model to its CUDA device first; grouped tables need one width")
        rows = [w.shape[0] for w in ws]
        buf = torch.empty(sum(rows), W, dtype=torch.float32, device=dev)
        grp = {"buf": buf, "rows": rows, "offsets": [sum(rows[:k]) for k in range(len(rows))], "m": None, "v": None}
        for k, e in enumerate(embeddings):
            o = grp["offsets"][k]
            buf[o:o + rows[k]].copy_(e.weight.data)
            e.weight = torch.nn.Parameter(buf[o:o + rows[k]], requires_grad=False)
            e.weight._rs_sink, e.weight._rs_group, e.weight._rs_field = self, grp, k
        self.groups.append(grp)
        return grp

    def record(self, weights, ids, dE):
        """weights: the looked-up tables, all of one group, in the column order of ids (N, F); dE (N, F, W)."""
        grp = weights[0]._rs_group
        for w in weights:
            if w._rs_group is not grp:
                raise RuntimeError("tables looked up together must belong to one fused group")
            if w.data_ptr() != grp["buf"].data_ptr() + grp["offsets"][w._rs_field] * grp["buf"].shape[1] * 4:
                raise RuntimeError("an embedding table was moved after fuse_embedding_updates(); call it after .to(device)")
        self.pending.append((grp, [w._rs_field for w in weights], ids, dE))

    def apply(self, opt):
        entries = self.pending
        if opt.kind != "sgd" or opt.weight_decay != 0.0:
            # Adam's moments and the decay term advance once per step: the lookups of several forwards into one group are
            # merged into one update over global rows (F = 1) on the summed gradient
            by_grp = {}
            for e in entries:
                by_grp.setdefault(id(e[0]), []).append(e)
            entries = [es[0] if len(es) == 1 else self._merged(es) for es in by_grp.values()]
        for grp, fields, ids, dE in entries:
            W = grp["buf"].shape[1]
            if fields is None:                  # merged entry: ids are global rows of the group's buffer
                F, offs = 1, None
            else:
                F, offs = len(fields), [grp["offsets"][f] for f in fields]
            segs = ops.dedup_sort(ids.reshape(-1, F), F, offs, sum(grp["rows"]), max_width=W)
            if opt.kind == "sgd":
                ops.segment_update(segs, ops.RS_UPD_SGD, W, F, dense=dE.reshape(-1, W), table=grp["buf"], lr=opt.lr, wd=opt.weight_decay)
            else:
                if grp["m"] is None:
                    grp["m"], grp["v"] = torch.zeros_like(grp["buf"]), torch.zeros_like(grp["buf"])
                ops.segment_update(segs, ops.RS_UPD_ADAM, W, F, dense=dE.reshape(-1, W), table=grp["buf"], m=grp["m"], v=grp["v"],
                                   lr=opt.lr, wd=opt.weight_decay, betas=opt.betas, eps=opt.eps, step=opt.step_count)
        self.pending.clear()

    @staticmethod
    def _merged(entries):
        grp, W = entries[0][0], entries[0][0]["buf"].shape[1]
        keys, rows = [], []
        for _, fields, ids, dE in entries:
            offs = torch.tensor([grp["offsets"][f] for f in fields], dtype=torch.int64, device=ids.device)
            keys.append((ids.reshape(-1, len(fields)) + offs).reshape(-1))
            rows.append(dE.reshape(-1, W))
        return grp, None, torch.cat(keys), torch.cat(rows)


class FusedRows:
    """Mixin: ``fuse_embedding_updates()`` + the apply_pending / clear_pending protocol FusedRowOptimizer drives."""
    _row_sink = None

    def _fused_groups(self):
        raise NotImplementedError

    def fuse_embedding_updates(self):
        if self._row_sink is None:
            self._row_sink = RowSink()
            for group in self._fused_groups():
                self._row_sink.add_group(group)
        return self

    def apply_pending(self, opt):
        if self._row_sink is not None:
            self._row_sink.apply(opt)

    def clear_pending(self):
        if self._row_sink is not None:
            self._row_sink.pending.clear()


class _FusedLookup(torch.autograd.Function):
    """weight[ids] whose backward records (ids, row gradients) for the fused row optimizer instead of a dense gradient"""

    @staticmethod
    def forward(ctx, anchor, weight, ids):
        ctx.weight = weight
        ctx.save_for_backward(ids)
        out = ops.gather_rows(ops.make_tables([weight.detach()]), ids.reshape(-1, 1))
        return out.view(*ids.shape, weight.shape[1])

    @staticmethod
    def backward(ctx, g):
        (ids,) = ctx.saved_tensors
        ctx.weight._rs_sink.record([ctx.weight], ids.reshape(-1, 1), g.contiguous().view(-1, 1, g.shape[-1]))
        return torch.zeros(1, device=g.device), None, None


class XEmbed(torch.autograd.Function):
    """Feature-vector front end: x (B,45) -> E (B, slots, D)  (reference model/deepfm.py:45-51 and siblings).

    slots: tuple of (col, ncols, kind); tables: one tensor per non-scalar slot, in slot order.
    Backward: id slots -> table_grads (sort/segment-reduce); bag slots -> rs_xembed_bag_bwd (two-pass fixed order).
    """

    @staticmethod
    def forward(ctx, x, slots, *tables):
        it = iter(tables)
        full = [(c, n, k, None if k == KIND_SCALAR else next(it).detach()) for c, n, k in slots]
        S = ops.make_xslots(full, tables[0].shape[1], x.shape[1])
        E = ops.xembed_fwd(S, x)
        ctx.slots = slots
        ctx.save_for_backward(x, *tables)
        return E

    @staticmethod
    def backward(ctx, dE):
        x, *tables = ctx.saved_tensors
        slots = ctx.slots
        dE = dE.contiguous()
        it = iter(tables)
        full = [(c, n, k, None if k == KIND_SCALAR else next(it).detach()) for c, n, k in slots]
        S = ops.make_xslots(full, tables[0].shape[1], x.shape[1])
        bag = ops.xembed_bag_bwd(S, x, dE, full) if any(k == KIND_BAG for _, _, k in slots) else [None] * len(slots)
        id_slots = [t for t, (_, _, k) in enumerate(slots) if k == KIND_ID]
        id_grads = {}
        if id_slots:
            ids = torch.stack([ops.xcol_to_ids(x, slots[t][0]) for t in id_slots], dim=1)
            g = dE[:, id_slots, :].contiguous() if len(id_slots) != len(slots) else dE
            for t, gw in zip(id_slots, table_grads(ids, g, [full[t][3].shape[0] for t in id_slots])):
                id_grads[t] = gw
        grads = []
        for t, (_, _, k) in enumerate(slots):
            if k == KIND_ID:
                grads.append(id_grads[t])
            elif k == KIND_BAG:
                grads.append(bag[t])
        return (None, None, *grads)


def six_slots():
    """[user, item, age, gender, occupation, movie] as the reference orders them (model/deepfm.py:54)."""
    return ((COL_USER, 1, KIND_ID), (COL_ITEM, 1, KIND_ID), (AGE[0], AGE[1], KIND_BAG), (GENDER[0], GENDER[1], KIND_BAG),
            (OCC[0], OCC[1], KIND_BAG), (GENRE[0], GENRE[1], KIND_BAG))


def five_slots():
    """[user, item, gender, occupation, movie]: the models that feed age as a raw scalar (model/widedeep.py:44-49)."""
    return ((COL_USER, 1, KIND_ID), (COL_ITEM, 1, KIND_ID), (GENDER[0], GENDER[1], KIND_BAG), (OCC[0], OCC[1], KIND_BAG),
            (GENRE[0], GENRE[1], KIND_BAG))


def stacked_features(x, user_w, item_w, gender_w, occupation_w, movie_w):
    """[e_user, e_item, age, e_gender, e_occupation, e_movie] -> (B, 5D+1): the stacking layer shared by
    model/widedeep.py:44-50, model/deepcross.py:60-66 and model/deepcrossing.py:56-63 (one fused lookup, one cat)."""
    E = XEmbed.apply(x, five_slots(), user_w, item_w, gender_w, occupation_w, movie_w)
    return torch.cat((E[:, :2].flatten(1), x[:, AGE[0]:AGE[0] + 1], E[:, 2:].flatten(1)), dim=1)


class _Interact(torch.autograd.Function):
    """Interaction over dense field embeddings E (B, F, D); `what` picks the output (rs_fields_fwd / rs_fields_bwd)."""

    @staticmethod
    def forward(ctx, E, what):
        E = E.contiguous()
        B, F, D = E.shape
        ctx.what = what
        ctx.save_for_backward(E)
        return ops.fields_fwd(ops.dummy_tables(F, D), B, E.device, dense_in=E, **{what: True})[what]

    @staticmethod
    def backward(ctx, g):
        (E,) = ctx.saved_tensors
        B, F, D = E.shape
        return ops.fields_bwd(ops.dummy_tables(F, D), B, E.device, dense_in=E, **{"g_" + ctx.what: g.contiguous()}), None


def fm_cross(E):
    """0.5*sum_d[(sum_f e)^2 - sum_f e^2] -> (B,)             model/deepfm.py:71-76"""
    return _Interact.apply(E, "cross")


def bi_interaction(E):
    """sum_{i<j} e_i*e_j -> (B, D)                             model/nfm.py:58-62"""
    return _Interact.apply(E, "bi")


def inner_products(E):
    """[<e_i,e_j>]_{i<j} -> (B, F(F-1)/2)                      model/pnn.py:61-66"""
    return _Interact.apply(E, "pairs")


class PairLookup(torch.autograd.Function):
    """Two id columns into two tables in one fused pass: MF dot (model/mf.py:24-26), GMF Hadamard
    (model/neuralcf.py:37-39) or the MLP-tower concat (model/neuralcf.py:43-46)."""

    @staticmethod
    def forward(ctx, wu, wi, u, i, what, anchor=None):
        ids = torch.stack([u, i], dim=1).contiguous()
        T = ops.make_tables([wu.detach(), wi.detach()])
        ctx.what, ctx.rows, ctx.fused = what, (wu.shape[0], wi.shape[0]), anchor is not None
        ctx.tables = (wu, wi)
        ctx.save_for_backward(ids)
        return ops.fields_fwd(T, ids.shape[0], ids.device, ids=ids, **{what: True})[what]

    @staticmethod
    def backward(ctx, g):
        (ids,) = ctx.saved_tensors
        wu, wi = ctx.tables
        T = ops.make_tables([wu.detach(), wi.detach()])
        dE = ops.fields_bwd(T, ids.shape[0], ids.device, ids=ids, **{"g_" + ctx.what: g.contiguous()})
        if ctx.fused:          # fused sparse mode: the row optimizer consumes (ids, dE); no table-sized gradient exists
            wu._rs_sink.record([wu, wi], ids, dE)
            return None, None, None, None, None, torch.zeros(1, device=g.device)
        if not (wu.requires_grad or wi.requires_grad):
            return None, None, None, None, None, None
        gu, gi = table_grads(ids, dE, list(ctx.rows))
        return gu, gi, None, None, None, None


def pair_lookup(wu, wi, u, i, what):
    sink = getattr(wu, "_rs_sink", None)
    if sink is not None and torch.is_grad_enabled():
        return PairLookup.apply(wu, wi, u, i, what, sink.anchor(wu.device))
    return PairLookup.apply(wu, wi, u, i, what, None)


class OuterPooled(torch.autograd.Function):
    """p = S^T S (D, D), the batch-collapsed outer product of PNN's "out" mode (reference model/pnn.py:69-72), on the
    tcgen05 tensor cores with a 3xTF32 split (rs_gemm_tn_3xtf32).  d loss / dS = S (G + G^T)."""

    @staticmethod
    def forward(ctx, S):
        S = S.contiguous()
        ctx.save_for_backward(S)
        return ops.gemm_tn(S, S)

    @staticmethod
    def backward(ctx, G):
        (S,) = ctx.saved_tensors
        return S @ (G + G.t())


class OuterProduct(torch.autograd.Function):
    """lp = W vec(s s^T) + b per sample, s = sum_f E[:, f] -- the PNN paper's outer-product layer with sum pooling (an
    extension: the reference's "out" mode is the batch-collapsed OuterPooled).  Forward and backward are one C-ABI call
    each (rs_pnn_outer_fwd / _bwd on tcgen05); every field row of a sample receives the same gradient dS."""

    @staticmethod
    def forward(ctx, E, W, b):
        lp, S = ops.pnn_outer_fwd(E, W, b)
        ctx.save_for_backward(S, W)
        ctx.F = E.shape[1]
        return lp

    @staticmethod
    def backward(ctx, g):
        S, W = ctx.saved_tensors
        dS, dW, db = ops.pnn_outer_bwd(S, g.contiguous(), W)
        return dS.unsqueeze(1).expand(-1, ctx.F, -1), dW, db


class FFMDense(torch.autograd.Function):
    """sum_{i<j} <T[i, field(j)], T[j, field(i)]> over dense T (B, F, NF, D)     model/ffm.py:61-82"""

    @staticmethod
    def forward(ctx, T, field_of):
        T = T.contiguous()
        ctx.field_of = field_of
        ctx.save_for_backward(T)
        return ops.ffm_dense_fwd(T, field_of)

    @staticmethod
    def backward(ctx, g):
        (T,) = ctx.saved_tensors
        return ops.ffm_dense_bwd(T, g.contiguous(), ctx.field_of), None


def first_order(module_user, module_item, linear, x):
    """user(1)[uid] + item(1)[iid] + Linear(43,1)(x[:,2:])     model/lr.py:24-25 and the wide terms of the others."""
    uid, iid = ops.xcol_to_ids(x, COL_USER), ops.xcol_to_ids(x, COL_ITEM)
    return lookup(module_user.weight, uid) + lookup(module_item.weight, iid) + linear(x[:, 2:])


RANK_CHUNK_ROWS = 1 << 18     # rows scored per forward while ranking the catalogue


def rank_catalogue(score_fn, num_users, num_items, k):
    """All users x all items -> (num_users, k) ranked item positions, as a numpy int64 array.

    ``score_fn(u0, u1)`` returns the scores of users [u0, u1) against items 0..num_items-1, user-major.  Users are
    scored a chunk at a time (one forward per ~RANK_CHUNK_ROWS rows instead of one per user) and every user's
    ``torch.topk(scores, k, dim=0)`` (reference model/din.py:63, model/neuralcf.py:69) is one CTA of rs_rank_segments."""
    import numpy as np
    if num_users == 0:
        return np.array([])
    step = max(1, RANK_CHUNK_ROWS // max(num_items, 1))
    out = []
    with torch.no_grad():
        for u0 in range(0, num_users, step):
            u1 = min(num_users, u0 + step)
            scores = score_fn(u0, u1).reshape(-1)
            out.append(ops.rank_segments(scores, k, seg_len=num_items))
    out = torch.cat(out).cpu().numpy()
    ops.check_status(scores.device)          # an out-of-range id raises IndexError, as nn.Embedding does on CPU
    return out


def history_scores(model, hist_list, num_items, device):
    """score_fn for DIN / DIEN: user u's history against every target item (reference model/din.py:58-62)."""
    try:
        hist_all = torch.tensor(hist_list)
        ragged = hist_all.dim() != 2
    except (ValueError, TypeError):
        ragged = True
    target = torch.arange(0, num_items, device=device)

    def score(u0, u1):
        if ragged:
            return torch.cat([model(torch.tensor(hist_list[u]).repeat(num_items, 1).to(device), target).reshape(-1)
                              for u in range(u0, u1)])
        hist = hist_all[u0:u1].to(device).repeat_interleave(num_items, dim=0)
        return model(hist, target.repeat(u1 - u0))
    return score


def topk_per_user(model, num_users, user_item, k, batched=True):
    """recommendation(): each user's rows of ``user_item`` scored and ranked (reference model/deepfm.py:85-95).

    The reference filters the frame once per user and runs one forward + topk per user.  Here the rows are grouped by
    user once (stable, so every user keeps the frame's row order -- the returned positions index that order), scored
    in large chunks, and ranked for all users by one rs_rank_segments launch.  ``batched=False`` keeps one forward per
    user for models whose output depends on the batch composition (PNN "out", model/pnn.py:72)."""
    import numpy as np
    device = next(model.parameters()).device
    uid = np.asarray(user_item["user_id"].values).astype(np.int64)
    keep = (uid >= 0) & (uid < num_users)
    grouped = bool(keep.all()) and bool((uid[1:] >= uid[:-1]).all())   # data.user_item() is already user-major
    if grouped:
        order = slice(None)
        counts = np.bincount(uid, minlength=num_users)
    else:
        order = np.flatnonzero(keep)
        order = order[np.argsort(uid[order], kind="stable")]
        counts = np.bincount(uid[order], minlength=num_users)
    values = np.asarray(user_item.values, dtype=np.float32)[order]
    n_rows = values.shape[0]
    seg = np.zeros(num_users + 1, dtype=np.int64)
    np.cumsum(counts, out=seg[1:])
    if num_users == 0:
        return np.array([])
    scores = []
    with torch.no_grad():
        if batched:
            for r0 in range(0, n_rows, RANK_CHUNK_ROWS):
                rows = torch.from_numpy(values[r0:r0 + RANK_CHUNK_ROWS]).to(device)
                scores.append(model(rows).reshape(-1))
        else:
            for u in range(num_users):
                rows = torch.from_numpy(values[seg[u]:seg[u + 1]]).to(device)
                scores.append(model(rows).reshape(-1))
        scores = torch.cat(scores) if scores else torch.empty(0, device=device)
        idx = ops.rank_segments(scores, k, seg_start=torch.from_numpy(seg).to(device), max_len=int(counts.max()))
    idx = idx.cpu().numpy()
    if device.type == "cuda":
        ops.check_status(device)             # an out-of-range id raises IndexError, as nn.Embedding does on CPU
    return idx
