"""Thin tensor-level wrappers over the C ABI (include/recsys_b200.h).  torch is plumbing only: it owns the
device memory and the stream; every op below is one call into librecsys_b200.so.  No CPU fallback."""
import ctypes as C

import os

import torch

from . import _lib
from ._lib import RS_MAX_FIELDS, RS_UPD_ADAM, RS_UPD_GRAD, RS_UPD_SGD  # noqa: F401

_status = {}
_launches = 0
PROFILE = None   # bench.py sets this to a list; ops then bracket their C-ABI call with CUDA events on the launching stream
NVTX = os.environ.get("RS_NVTX", "0") == "1"   # every C-ABI call and every exchange phase becomes an NVTX range (nsys / ncu --nvtx)


class _timed:
    def __init__(self, name):
        self.name = name

    def __enter__(self):
        if NVTX:
            torch.cuda.nvtx.range_push(self.name)
        if PROFILE is not None:
            self.a = torch.cuda.Event(enable_timing=True)
            self.a.record()

    def __exit__(self, *exc):
        if NVTX:
            torch.cuda.nvtx.range_pop()
        if PROFILE is not None:
            b = torch.cuda.Event(enable_timing=True)
            b.record()
            PROFILE.append((self.name, self.a, b))


def launches():
    """Number of C-ABI calls that launched kernels since import (bench.py reports it)."""
    return _launches


def _count(n=1):
    global _launches
    _launches += n


def _need_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError("deeplearningrecommendationsystem_b200 ops need CUDA tensors (there is no CPU fallback)")


def _p(t):
    return None if t is None else t.data_ptr()


def _f32(t):
    if t is None:
        return None
    if t.dtype != torch.float32:
        raise TypeError(f"expected float32, got {t.dtype}")
    return t.contiguous()


def _i64(t):
    if t.dtype != torch.int64:
        raise TypeError(f"ids must be int64, got {t.dtype}")
    return t.contiguous()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def status_word(device):
    key = torch.device(device).index if torch.device(device).index is not None else torch.cuda.current_device()
    if key not in _status:
        _status[key] = torch.zeros(1, dtype=torch.int32, device=f"cuda:{key}")
    return _status[key]


def check_status(device=None):
    """Synchronising check of the out-of-range-id flag; raises IndexError like nn.Embedding does on CPU."""
    w = status_word(device if device is not None else torch.cuda.current_device())
    v = int(w.item())
    if v:
        w.zero_()
        if v & 16:
            raise RuntimeError("row exchange: an owner was asked for more rows than its receive capacity "
                               "(raise recv_slack of the DeviceRowExchange); the step's update is incomplete")
        if v & 8:
            raise RuntimeError("dien_negatives: a slot found no item distinct from its positive in 65536 attempts")
        raise IndexError("index out of range in embedding lookup")


def make_tables(weights, width=None):
    """rs_tables from a list of (rows_f, W) fp32 CUDA tensors (one per field)."""
    T = _lib.rs_tables()
    if len(weights) > RS_MAX_FIELDS:
        raise ValueError(f"at most {RS_MAX_FIELDS} fields")
    T.num_fields = len(weights)
    T.width = int(width if width is not None else weights[0].shape[1])
    for f, w in enumerate(weights):
        _need_cuda(w)
        if w.dtype != torch.float32 or not w.is_contiguous() or w.shape[1] != T.width:
            raise ValueError("tables must be contiguous float32 (rows, width)")
        T.base[f] = w.data_ptr()
        T.rows[f] = w.shape[0]
    return T


def tables_from_concat(weight, offsets, rows):
    """rs_tables over ONE concatenated (total_rows, W) tensor: field f starts at row offsets[f]."""
    T = _lib.rs_tables()
    T.num_fields = len(rows)
    T.width = weight.shape[1]
    base = weight.data_ptr()
    for f, (o, r) in enumerate(zip(offsets, rows)):
        T.base[f] = base + int(o) * T.width * 4
        T.rows[f] = int(r)
    return T


def dummy_tables(F, D):
    T = _lib.rs_tables()
    T.num_fields, T.width = F, D
    return T


def gather_rows(T, ids):
    """out[..., f, :] = table_f[ids[..., f]]; ids (B, F) -> (B, F, W).  Bit-exact row copy."""
    ids = _i64(ids)
    _need_cuda(ids)
    B = ids.numel() // T.num_fields
    out = torch.empty(B, T.num_fields, T.width, dtype=torch.float32, device=ids.device)
    if B == 0:
        return out
    with _timed(f"gather_rows[w{T.width}]"):
        _lib.check(_lib.load().rs_gather_rows(C.byref(T), ids.data_ptr(), B, out.data_ptr(), status_word(ids.device).data_ptr(),
                                              _stream()), "rs_gather_rows")
    _count()
    return out


def fields_fwd(T, B, device, ids=None, dense_in=None, cross=False, bi=False, pairs=False, concat=False, stash=False,
               dot2=False, had2=False):
    """Fused lookup + interaction forward.  Returns a dict of the requested outputs."""
    F, D = T.num_fields, T.width
    io = _lib.rs_fields_io()
    keep = []
    if ids is not None:
        ids = _i64(ids)
        _need_cuda(ids)
        io.ids = ids.data_ptr()
    else:
        dense_in = _f32(dense_in)
        _need_cuda(dense_in)
        io.dense_in = dense_in.data_ptr()
    out = {}

    def alloc(name, *shape):
        t = torch.empty(*shape, dtype=torch.float32, device=device)
        out[name] = t
        setattr(io, name, t.data_ptr())

    if cross:
        alloc("cross", B)
    if bi:
        alloc("bi", B, D)
    if pairs:
        alloc("pairs", B, F * (F - 1) // 2)
    if concat:
        alloc("concat", B, F * D)
    if stash:
        alloc("stash", B, F, D)
    if dot2:
        alloc("dot2", B)
    if had2:
        alloc("had2", B, D)
    if B == 0:
        return out
    with _timed("fields_fwd"):
        _lib.check(_lib.load().rs_fields_fwd(C.byref(T), C.byref(io), B, status_word(device).data_ptr(), _stream()), "rs_fields_fwd")
    _count()
    del keep
    return out


def fields_bwd(T, B, device, ids=None, dense_in=None, g_cross=None, g_bi=None, g_pairs=None, g_concat=None, g_dot2=None,
               g_had2=None):
    """dE (B, F, D): gradient of the interaction outputs w.r.t. the field embeddings."""
    F, D = T.num_fields, T.width
    g = _lib.rs_fields_grad()
    if ids is not None:
        ids = _i64(ids)
        g.ids = ids.data_ptr()
    else:
        dense_in = _f32(dense_in)
        g.dense_in = dense_in.data_ptr()
    ups = dict(g_cross=_f32(g_cross), g_bi=_f32(g_bi), g_pairs=_f32(g_pairs), g_concat=_f32(g_concat), g_dot2=_f32(g_dot2),
               g_had2=_f32(g_had2))
    for k, t in ups.items():
        _need_cuda(t)
        setattr(g, k, _p(t))
    dE = torch.empty(B, F, D, dtype=torch.float32, device=device)
    g.dE = dE.data_ptr()
    if B == 0:
        return dE
    _lib.check(_lib.load().rs_fields_bwd(C.byref(T), C.byref(g), B, _stream()), "rs_fields_bwd")
    _count()
    return dE


def ffm_fwd(T, ids, D, want_stash=True, peer=None, split_mask=0):
    """cross (B,), stash (B, F, F*D) | None for an F-field FFM whose table rows are (F, D).
    peer=(world, direct_mask, shard_ptrs, total_rows): row-sharded tables, the fields of direct_mask are read straight from
    the owning rank's shard over NVLink (ids of those fields are GLOBAL rows) -- rs_ffm_fwd_peer.
    split_mask != 0 (with peer): returns (cross, stash_rest (B, F - k, W), stash_split (B, k, W)) -- the Jacobian rows of the
    k fields in split_mask are written to their own tensor (the row-sharded tables), the others' (replicated tables) to
    stash_rest."""
    ids = _i64(ids)
    _need_cuda(ids)
    F = T.num_fields
    B = ids.numel() // F
    cross = torch.empty(B, dtype=torch.float32, device=ids.device)
    k = bin(split_mask & ((1 << F) - 1)).count("1") if split_mask else 0
    stash = torch.empty(B, F - k, F * D, dtype=torch.float32, device=ids.device) if want_stash else None
    stash2 = torch.empty(B, k, F * D, dtype=torch.float32, device=ids.device) if (want_stash and k) else None
    if B == 0:
        return (cross, stash, stash2) if split_mask else (cross, stash)
    PT = None
    if peer is not None:
        PT = _lib.rs_peer_tables()
        PT.world, PT.direct_mask, PT.total_rows = int(peer[0]), int(peer[1]), int(peer[3])
        for r, ptr in enumerate(peer[2]):
            PT.shard[r] = int(ptr)
        if stash2 is not None:
            PT.split_mask, PT.stash_split = int(split_mask), stash2.data_ptr()
        PT = C.byref(PT)
    with _timed("ffm_fwd"):
        _lib.check(_lib.load().rs_ffm_fwd_peer(C.byref(T), ids.data_ptr(), B, D, PT, cross.data_ptr(), _p(stash),
                                               status_word(ids.device).data_ptr(), _stream()), "rs_ffm_fwd")
    _count()
    return (cross, stash, stash2) if split_mask else (cross, stash)


def ffm_fwd_train(T, ids, D, cold_mask):
    """Training forward of the stash-free FFM step: cross (B,) and the cold-slice stash (B, F, nC, D) -- slot i of the rows
    of the nC fields flagged in cold_mask, for every lookup (b, i) -- that ffm_bwd_update consumes (rs_ffm_fwd_train)."""
    ids = _i64(ids)
    _need_cuda(ids)
    F = T.num_fields
    B = ids.numel() // F
    nC = bin(cold_mask & ((1 << F) - 1)).count("1")
    cross = torch.empty(B, dtype=torch.float32, device=ids.device)
    mini = torch.empty(B, F, nC, D, dtype=torch.float32, device=ids.device) if nC else None
    if B == 0:
        return cross, mini
    with _timed("ffm_fwd"):
        _lib.check(_lib.load().rs_ffm_fwd_train(C.byref(T), ids.data_ptr(), B, D, int(cold_mask), cross.data_ptr(), _p(mini),
                                                status_word(ids.device).data_ptr(), _stream()), "rs_ffm_fwd_train")
    _count()
    return cross, mini


def _field_of(field_of):
    return (C.c_int32 * len(field_of))(*field_of)


def ffm_dense_fwd(Tin, field_of):
    Tin = _f32(Tin)
    _need_cuda(Tin)
    B, F, NF, D = Tin.shape
    cross = torch.empty(B, dtype=torch.float32, device=Tin.device)
    if B == 0:
        return cross
    _lib.check(_lib.load().rs_ffm_dense_fwd(Tin.data_ptr(), B, F, NF, D, _field_of(field_of), cross.data_ptr(), _stream()),
               "rs_ffm_dense_fwd")
    _count()
    return cross


def ffm_dense_bwd(Tin, g_cross, field_of):
    Tin, g_cross = _f32(Tin), _f32(g_cross)
    B, F, NF, D = Tin.shape
    dT = torch.empty_like(Tin)
    if B == 0:
        return dT
    _lib.check(_lib.load().rs_ffm_dense_bwd(Tin.data_ptr(), g_cross.data_ptr(), B, F, NF, D, _field_of(field_of), dT.data_ptr(),
                                            _stream()), "rs_ffm_dense_bwd")
    _count()
    return dT


class Segments:
    """Result of dedup_sort: device arrays carved out of one workspace tensor (kept alive here)."""

    def __init__(self, ws, seg, n, device):
        self.ws, self.seg, self.n, self.device = ws, seg, n, device
        self.ready = None

    def _view(self, ptr, count, dtype):
        off = ptr - self.ws.data_ptr()
        size = torch.empty(0, dtype=dtype).element_size()
        return self.ws[off:off + count * size].view(dtype)

    @property
    def n_uniq(self):
        return int(self._view(self.seg.n_uniq, 1, torch.int32).item())

    def uniq(self):
        return self._view(self.seg.uniq, self.n, torch.int64)[: self.n_uniq]

    def inverse(self):
        return self._view(self.seg.inverse, self.n, torch.int32)

    def counts(self):
        return self._view(self.seg.counts, self.n, torch.int32)[: self.n_uniq]

    def sorted_pos(self):
        return self._view(self.seg.sorted_pos, self.n, torch.int32)


_partial_cache = {}
_seg_memo = {}
_MEMO_SLOTS = 4      # memoised dedup results per device (each owns its workspace)


def _partial_buffer(device, n, width):
    """Scratch for chunk partial sums: 2*(n/RS_CHUNK + 2) rows of `width` floats, cached per (device, size)."""
    need = 2 * (n // _lib.RS_CHUNK + 2) * width
    key = (device, n)
    buf = _partial_cache.get(key)
    if buf is None or buf.numel() < need:
        buf = torch.empty(need, dtype=torch.float32, device=device)
        _partial_cache[key] = buf
    return buf


def dedup_sort(ids, F=1, row_offset=None, total_rows=None, max_width=1, reuse_workspace=True, shard=None, n_valid=None):
    """Stable sort of the lookups by global table row + segment/chunk boundaries (no host sync).

    shard=(world, rows_per_rank): owner-major keys for row-sharded tables (rs_dedup_sort_ex); n_valid: int32 device
    scalar, only the first n_valid ids are real (fixed-capacity receive lists).  Both bypass the memo.

    The result depends only on (ids, F, row_offset, total_rows), so a second request for the SAME ids tensor (same
    storage, same version counter -- e.g. the FM and the FFM model stepping on one batch) returns the memoised
    segments instead of sorting again.  `max_width` only sizes the partial-sum scratch, which is attached lazily.
    """
    ids = _i64(ids)
    _need_cuda(ids)
    n = ids.numel()
    lib = _lib.load()
    if shard is not None or n_valid is not None:
        reuse_workspace = False
    memo_key = (ids.data_ptr(), ids._version, n, F, tuple(int(o) for o in row_offset) if row_offset is not None else None,
                int(total_rows)) if reuse_workspace else None
    slots = _seg_memo.setdefault(ids.device, []) if reuse_workspace else None
    segs = None
    if reuse_workspace:
        for i, (k, sg, ref) in enumerate(slots):
            if k == memo_key and ref is ids:
                segs = sg
                slots.append(slots.pop(i))          # most recently used last
                if segs.ready is not None:          # produced on another stream (prefetch_dedup): order after it
                    torch.cuda.current_stream().wait_event(segs.ready)
                break
    if segs is None:
        nbytes = C.c_size_t(0)
        _lib.check(lib.rs_dedup_workspace_bytes(n, 1, C.byref(nbytes)), "rs_dedup_workspace_bytes")
        ws = None
        if reuse_workspace and len(slots) >= _MEMO_SLOTS:     # recycle the least recently used slot's workspace
            _, old, _ = slots.pop(0)
            if old.ws.numel() >= nbytes.value:
                ws = old.ws
        if ws is None:
            ws = torch.empty(nbytes.value, dtype=torch.uint8, device=ids.device)
        seg = _lib.rs_segments()
        offs = None
        if row_offset is not None:
            offs = (C.c_int64 * F)(*[int(o) for o in row_offset])
        opts = None
        if shard is not None or n_valid is not None:
            opts = _lib.rs_dedup_opts()
            opts.n_valid = _p(n_valid)
            opts.shard_world, opts.shard_rows = (int(shard[0]), int(shard[1])) if shard is not None else (0, 0)
            opts = C.byref(opts)
        with _timed("dedup_sort"):
            _lib.check(lib.rs_dedup_sort_ex(ids.data_ptr(), n, F, offs, int(total_rows), opts, ws.data_ptr(), ws.numel(), C.byref(seg),
                                            status_word(ids.device).data_ptr(), _stream()), "rs_dedup_sort")
        _count(10)
        segs = Segments(ws, seg, n, ids.device)
        if reuse_workspace:
            slots.append((memo_key, segs, ids))
        if _prefetching:
            segs.ready = torch.cuda.Event()
            segs.ready.record()
    part = _partial_buffer(ids.device, n, int(max_width)) if reuse_workspace else \
        torch.empty(2 * (n // _lib.RS_CHUNK + 2) * int(max_width), dtype=torch.float32, device=ids.device)
    segs.partial = part
    segs.seg.partial = part.data_ptr()
    segs.seg.partial_floats = part.numel()
    return segs


def invalidate_dedup(device=None):
    """Forget the memoised sorts (of `device`, or of every device).  The memo recognises an id tensor by (storage pointer,
    version counter, identity): writes that bypass the version counter -- `ids.data.copy_()`, a kernel or a CUDA-graph
    replay writing through the pointer -- are invisible to it, so call this after such a write if the same tensor object
    is then handed to an op again eagerly."""
    if device is None:
        _seg_memo.clear()
    else:
        _seg_memo.pop(torch.device(device), None)


def attach_partial(segs, width):
    """(Re)attach the chunk-partial scratch for rows of `width` floats to finished segments."""
    part = _partial_buffer(segs.device, segs.n, int(width))
    segs.partial = part
    segs.seg.partial = part.data_ptr()
    segs.seg.partial_floats = part.numel()
    return segs


def block_segments(segs, n_uniq, width):
    """Re-use the segments of a dedup over global keys for the rows of the fetched block: the j-th distinct key IS block
    row j, so only the row ids change (rs_segments_relabel, once) -- the stable order, segment and chunk boundaries are
    identical to what sorting the block-local ids again would give."""
    if not getattr(segs, "relabelled", False):
        _lib.check(_lib.load().rs_segments_relabel(C.byref(segs.seg), segs.n, _stream()), "rs_segments_relabel")
        _count()
        segs.relabelled = True
    part = _partial_buffer(segs.device, segs.n, int(width))
    segs.partial = part
    segs.seg.partial = part.data_ptr()
    segs.seg.partial_floats = part.numel()
    return segs


_prefetching = False
_side_streams = {}


def prefetch_dedup(ids, F=1, row_offset=None, total_rows=None):
    """Run rs_dedup_sort for `ids` on a side stream NOW (it depends only on the ids), so the sort overlaps the forward
    kernels; the later dedup_sort() call on the main stream finds the memoised result and waits on its event."""
    global _prefetching
    dev = ids.device
    side = _side_streams.get(dev)
    if side is None:
        side = _side_streams[dev] = torch.cuda.Stream(device=dev)
    side.wait_stream(torch.cuda.current_stream(dev))      # ids may have just been produced on the main stream
    _prefetching = True
    try:
        with torch.cuda.stream(side):
            dedup_sort(ids, F, row_offset, total_rows, max_width=1)
    finally:
        _prefetching = False


def make_routes(starts, bases, row0s, dyn_start=None, dyn_row0=None, cap_rows=0, self_index=-1):
    """rs_routes: logical rows [starts[k], starts[k+1]) go to bases[k] (device pointer, peer-mapped or local) at row
    offset row0s[k].  len(starts) == len(bases) + 1.  dyn_start / dyn_row0: device addresses of the same two arrays
    (int64) when they only exist on the device (host-sync-free sharded step); starts / row0s are then ignored."""
    R = _lib.rs_routes()
    R.n = len(bases)
    for k, b in enumerate(bases):
        R.base[k] = int(b)
    if dyn_start is None:
        for k, (s0, r0) in enumerate(zip(starts, row0s)):
            R.start[k], R.row0[k] = int(s0), int(r0)
        R.start[R.n] = int(starts[-1])
    else:
        R.dyn_start, R.dyn_row0 = int(dyn_start), int(dyn_row0)
    R.cap_rows = int(cap_rows)
    R.self = int(self_index)
    return R


def make_shard(world, rank, rows_per_rank, cap_req, cap_recv, req_ptrs, ctl_ptrs, direct=()):
    """rs_shard: the per-exchange constants + the peer-mapped request / control buffers of every rank.
    direct: global-row ranges [(lo, hi), ...] whose rows are read by the forward kernel itself (not fetched)."""
    S = _lib.rs_shard()
    S.world, S.rank, S.rows_per_rank, S.cap_req, S.cap_recv = world, rank, int(rows_per_rank), int(cap_req), int(cap_recv)
    for k in range(world):
        S.req[k], S.ctl[k] = int(req_ptrs[k]), int(ctl_ptrs[k])
    if len(direct) > _lib.RS_MAX_DIRECT:
        raise ValueError(f"at most {_lib.RS_MAX_DIRECT} direct row ranges")
    S.n_direct = len(direct)
    for k, (lo, hi) in enumerate(direct):
        S.direct_lo[k], S.direct_hi[k] = int(lo), int(hi)
    return S


def shard_post(S, segs):
    """requester: request lists + counts written straight into the owners' buffers (follow with a cross-rank barrier)"""
    with _timed("shard_post"):
        _lib.check(_lib.load().rs_shard_post(C.byref(S), C.byref(segs.seg), segs.n, status_word(segs.device).data_ptr(), _stream()),
                   "rs_shard_post")
    _count()


def shard_collect(S, recv_local, m_total, recv_skip=None):
    """owner: prefix of the received counts, compact receive list (first m_total entries of recv_local; recv_skip flags the
    requests that lie in a direct range), gradient offsets sent back to the requesters"""
    _need_cuda(recv_local, m_total)
    with _timed("shard_collect"):
        _lib.check(_lib.load().rs_shard_collect(C.byref(S), recv_local.data_ptr(), _p(recv_skip), m_total.data_ptr(),
                                                status_word(recv_local.device).data_ptr(), _stream()), "rs_shard_collect")
    _count()


def shard_serve(S, table, recv_local, block_ptrs, cap_block_rows, skip=None):
    """owner: table[recv_local[i]] -> the requesters' blocks over NVLink (follow with a cross-rank barrier); rows flagged in
    `skip` (uint8) are not copied"""
    _need_cuda(table, recv_local)
    ptrs = (C.c_void_p * S.world)(*[int(p) for p in block_ptrs])
    with _timed(f"shard_serve[w{table.shape[1]}]"):
        _lib.check(_lib.load().rs_shard_serve(C.byref(S), table.data_ptr(), table.shape[0], table.shape[1], recv_local.data_ptr(), _p(skip), ptrs,
                                              int(cap_block_rows), status_word(table.device).data_ptr(), _stream()), "rs_shard_serve")
    _count()


def gather_rows_peer(table, idx, routes):
    """Owner side of the fused gather + all-to-all: table[idx[i]] is stored straight into the requesting rank's block
    through its peer-mapped pointer (routes).  Follow with a cross-rank barrier."""
    _need_cuda(table, idx)
    idx = _i64(idx)
    if idx.numel() == 0:
        return
    with _timed(f"gather_rows_peer[w{table.shape[1]}]"):
        _lib.check(_lib.load().rs_gather_rows_peer(table.data_ptr(), table.shape[0], table.shape[1], idx.data_ptr(), idx.numel(),
                                                   C.byref(routes), status_word(table.device).data_ptr(), _stream()),
                   "rs_gather_rows_peer")
    _count()


def segment_update(segs, mode, width, F, stash=None, scale=None, dense=None, table=None, m=None, v=None, dense_grad=None,
                   lr=0.0, wd=0.0, betas=(0.9, 0.999), eps=1e-8, step=1, grad_routes=None, tag="", half_sm=False):
    """Segment-reduce the per-lookup row gradients (scale*stash + dense) and apply `mode` to the touched rows."""
    u = _lib.rs_update()
    u.mode, u.width, u.F = mode, width, F
    stash, scale, dense = _f32(stash), _f32(scale), _f32(dense)
    u.scale_width = 1 if (scale is None or scale.numel() * F == segs.n) else width
    for name, t in (("stash", stash), ("scale", scale), ("dense", dense), ("table", table), ("m", m), ("v", v),
                    ("dense_grad", dense_grad)):
        _need_cuda(t)
        if t is not None and (t.dtype != torch.float32 or not t.is_contiguous()):
            raise ValueError(f"{name} must be contiguous float32")
        setattr(u, name, _p(t))
    u.lr, u.wd, u.beta1, u.beta2, u.eps, u.step = lr, wd, betas[0], betas[1], eps, step
    if grad_routes is not None:
        u.grad_routes = C.pointer(grad_routes)
    u.half_sm = 1 if half_sm else 0
    with _timed(f"segment_update{tag}[w{width}]"):
        _lib.check(_lib.load().rs_segment_update(C.byref(segs.seg), segs.n, C.byref(u), _stream()), "rs_segment_update")
    _count(2)


_ffm_bwd_ws = {}


def ffm_bwd_update(T, ids, D, segs, g_cross, table, lr, wd=0.0, cold_mask=0, cold_stash=None, tag=""):
    """FFM backward + fused SGD row update rebuilt from the table (rs_ffm_bwd_update): no full Jacobian stash.
    T: rs_tables over `table` (the concatenated (total_rows, F*D) tensor), ids (B, F) the batch the forward ran on,
    segs = dedup_sort(ids, ..., max_width=F*D), g_cross (B,) = dL/dcross, (cold_mask, cold_stash) as given to / returned by
    ffm_fwd_train.  The table must be unchanged since the forward."""
    ids, g_cross = _i64(ids), _f32(g_cross)
    _need_cuda(ids, g_cross, table, cold_stash)
    F = T.num_fields
    B = ids.numel() // F
    if B == 0:
        return
    lib = _lib.load()
    nbytes = C.c_size_t(0)
    _lib.check(lib.rs_ffm_bwd_ws_bytes(B * F, B, F * D, C.byref(nbytes)), "rs_ffm_bwd_ws_bytes")
    key = (ids.device, B * F, F * D)
    ws = _ffm_bwd_ws.get(key)
    if ws is None or ws.numel() < nbytes.value:
        _ffm_bwd_ws.clear()                                  # one shape at a time: the buffer is ~half a stash
        ws = _ffm_bwd_ws[key] = torch.empty(nbytes.value, dtype=torch.uint8, device=ids.device)
    u = _lib.rs_update()
    u.mode, u.width, u.F, u.scale_width = RS_UPD_SGD, F * D, F, 1
    u.scale, u.table = g_cross.data_ptr(), table.data_ptr()
    u.lr, u.wd, u.step = lr, wd, 1
    with _timed(f"ffm_bwd_update{tag}"):
        _lib.check(lib.rs_ffm_bwd_update(C.byref(T), ids.data_ptr(), B, D, int(cold_mask), _p(cold_stash), C.byref(segs.seg), C.byref(u), ws.data_ptr(), ws.numel(),
                                         status_word(ids.device).data_ptr(), _stream()), "rs_ffm_bwd_update")
    _count(5)


def replica_sgd(w_ptrs, g_ptrs, numel, world, rank, lr, wd=0.0):
    """Replicated table: sum the ranks' dense gradients in rank order, SGD step, result stored into every rank's copy
    (rs_replica_sgd).  w_ptrs / g_ptrs: per-rank device addresses (symmetric memory).  Barriers before and after are the
    caller's."""
    W = (C.c_void_p * world)(*[int(p) for p in w_ptrs])
    G = (C.c_void_p * world)(*[int(p) for p in g_ptrs])
    with _timed("replica_sgd"):
        _lib.check(_lib.load().rs_replica_sgd(W, G, int(numel), world, rank, lr, wd, _stream()), "rs_replica_sgd")
    _count()


def replica_slice(numel, world, rank):
    """(lo, hi) in floats of the elements rank `rank` updates in replica_sgd / replica_update (float4 slices,
    per = ceil(numel / 4 / world))"""
    n4 = int(numel) // 4
    per = (n4 + world - 1) // world
    lo4 = min(per * rank, n4)
    return lo4 * 4, min(lo4 + per, n4) * 4


def mark_rows(segs, touched, rows):
    """touched[uniq[j]] = 1 for the distinct rows of a finished sort (rs_mark_rows; the count stays on the device).
    touched: uint8 (rows,), zeroed by the caller."""
    _need_cuda(touched)
    if touched.dtype != torch.uint8 or not touched.is_contiguous() or touched.numel() < rows:
        raise ValueError("touched must be a contiguous uint8 tensor of at least `rows` flags")
    with _timed("mark_rows"):
        _lib.check(_lib.load().rs_mark_rows(C.byref(segs.seg), segs.n, touched.data_ptr(), int(rows),
                                            status_word(touched.device).data_ptr(), _stream()), "rs_mark_rows")
    _count()


def replica_update(w_ptrs, g_ptrs, flag_ptrs, numel, width, world, rank, kind, lr, wd=0.0, m=None, v=None, betas=(0.9, 0.999),
                   eps=1e-8, step=1):
    """Replicated table, lazy row update (rs_replica_update): rows flagged by some rank (flag_ptrs: every rank's uint8
    touched array) take an SGD ("sgd") or Adam ("adam") step on the rank-ordered sum of the ranks' gradients, stored into
    every rank's copy; the others keep their bits.  m / v: this rank's moment slices, replica_slice() floats from its lo.
    Barriers before and after are the caller's."""
    if kind not in ("sgd", "adam"):
        raise ValueError("kind must be 'sgd' or 'adam'")
    u = _lib.rs_update()
    u.mode, u.width = (RS_UPD_SGD if kind == "sgd" else RS_UPD_ADAM), int(width)
    if kind == "adam":
        lo, hi = replica_slice(numel, world, rank)
        for name, t in (("m", m), ("v", v)):
            if t is None or t.dtype != torch.float32 or not t.is_contiguous() or t.numel() != hi - lo:
                raise ValueError(f"{name} must be a contiguous float32 slice of {hi - lo} elements")
            if hi > lo:
                _need_cuda(t)
                setattr(u, name, t.data_ptr())
    u.lr, u.wd, u.beta1, u.beta2, u.eps, u.step = lr, wd, betas[0], betas[1], eps, step
    W = (C.c_void_p * world)(*[int(p) for p in w_ptrs])
    G = (C.c_void_p * world)(*[int(p) for p in g_ptrs])
    T = (C.c_void_p * world)(*[int(p) for p in flag_ptrs])
    with _timed(f"replica_update[{kind}]"):
        _lib.check(_lib.load().rs_replica_update(W, G, T, int(numel), world, rank, C.byref(u), _stream()), "rs_replica_update")
    _count()


def adam_dense(p, g, m, v, step, lr=1e-3, wd=0.0, betas=(0.9, 0.999), eps=1e-8):
    _need_cuda(p, g, m, v)
    _lib.check(_lib.load().rs_adam_dense(p.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr(), p.numel(), lr, wd, betas[0],
                                         betas[1], eps, step, _stream()), "rs_adam_dense")
    _count()


def make_xslots(slots, width, xcols):
    """slots: list of (col, ncols, kind, table|None)."""
    S = _lib.rs_xslots()
    S.num_slots, S.width, S.xcols = len(slots), width, xcols
    for t, (col, ncols, kind, table) in enumerate(slots):
        S.col[t], S.ncols[t], S.kind[t] = col, ncols, kind
        if table is not None:
            _need_cuda(table)
            S.table[t] = table.data_ptr()
            S.rows[t] = table.shape[0]
    return S


def xembed_fwd(S, x):
    x = _f32(x)
    _need_cuda(x)
    B = x.shape[0]
    E = torch.empty(B, S.num_slots, S.width, dtype=torch.float32, device=x.device)
    if B == 0:
        return E
    _lib.check(_lib.load().rs_xembed_fwd(C.byref(S), x.data_ptr(), B, E.data_ptr(), status_word(x.device).data_ptr(), _stream()),
               "rs_xembed_fwd")
    _count()
    return E


def xembed_bag_bwd(S, x, dE, slots):
    """-> list (per slot) of dW (ncols, W) for bag slots, None otherwise.  Fixed-order two-pass reduction."""
    x, dE = _f32(x), _f32(dE)
    B = x.shape[0]
    if B == 0:
        return [torch.zeros(nc, S.width, dtype=torch.float32, device=x.device) if kind == 1 else None for _, nc, kind, _ in slots]
    lib = _lib.load()
    nbytes = C.c_size_t(0)
    _lib.check(lib.rs_xembed_bag_ws_bytes(C.byref(S), B, C.byref(nbytes)), "rs_xembed_bag_ws_bytes")
    ws = torch.empty(nbytes.value // 4 + 1, dtype=torch.float32, device=x.device)
    outs, ptrs = [], (C.c_void_p * S.num_slots)()
    for t, (col, ncols, kind, table) in enumerate(slots):
        if kind == 1:
            w = torch.empty(ncols, S.width, dtype=torch.float32, device=x.device)
            outs.append(w)
            ptrs[t] = w.data_ptr()
        else:
            outs.append(None)
    _lib.check(lib.rs_xembed_bag_bwd(C.byref(S), x.data_ptr(), dE.data_ptr(), B, ptrs, ws.data_ptr(), nbytes.value, _stream()),
               "rs_xembed_bag_bwd")
    _count(2)
    return outs


def xcol_to_ids(x, col):
    x = _f32(x)
    _need_cuda(x)
    ids = torch.empty(x.shape[0], dtype=torch.int64, device=x.device)
    if x.shape[0] == 0:
        return ids
    _lib.check(_lib.load().rs_xcol_to_ids(x.data_ptr(), x.shape[0], x.shape[1], col, ids.data_ptr(), _stream()), "rs_xcol_to_ids")
    _count()
    return ids


def sigmoid_bce(logit, y, want_grad=True, bias=None, want_gsum=False):
    """pred, mean BCE loss (0-d tensor), d loss / d logit -- one fused pass + fixed-order reduction.
    bias (1-element tensor): the logit is `logit + bias` (the models' last step, folded in); want_gsum: also return
    sum(d loss / d logit) (the bias gradient, shape (1,)) as a fourth value."""
    logit, y = _f32(logit).view(-1), _f32(y).view(-1)
    _need_cuda(logit, y, bias)
    B = logit.numel()
    pred = torch.empty_like(logit)
    g = torch.empty_like(logit) if want_grad else None
    loss = torch.empty((), dtype=torch.float32, device=logit.device)
    gsum = torch.empty(1, dtype=torch.float32, device=logit.device) if want_gsum else None
    ws = torch.empty(2048, dtype=torch.float32, device=logit.device)
    _lib.check(_lib.load().rs_sigmoid_bce_bias(logit.data_ptr(), _p(_f32(bias)), y.data_ptr(), B, pred.data_ptr(), _p(g), loss.data_ptr(),
                                               _p(gsum), ws.data_ptr(), _stream()), "rs_sigmoid_bce")
    _count(2)
    return (pred, loss, g, gsum) if want_gsum else (pred, loss, g)


def gru_fwd(gi, w_hh, b_hh, want_gates=True):
    """gi (B, L, 3H) = x.W_ih^T + b_ih  ->  h_all (B, L, H), gates (B, L, 4H) | None."""
    gi, w_hh, b_hh = _f32(gi), _f32(w_hh), _f32(b_hh)
    _need_cuda(gi, w_hh, b_hh)
    B, L, H3 = gi.shape
    H = H3 // 3
    h_all = torch.empty(B, L, H, dtype=torch.float32, device=gi.device)
    gates = torch.empty(B, L, 4 * H, dtype=torch.float32, device=gi.device) if want_gates else None
    if B == 0:
        return h_all, gates
    with _timed("gru_fwd"):
        _lib.check(_lib.load().rs_gru_fwd(gi.data_ptr(), B, L, H, w_hh.data_ptr(), b_hh.data_ptr(), h_all.data_ptr(), _p(gates),
                                          _stream()), "rs_gru_fwd")
    _count()
    return h_all, gates


def gru_bwd(w_hh, h_all, gates, g_h_all=None, g_h_last=None):
    """-> d_gi, d_gh (B, L, 3H)."""
    B, L, H = h_all.shape
    g_h_all, g_h_last = _f32(g_h_all), _f32(g_h_last)
    d_gi = torch.empty(B, L, 3 * H, dtype=torch.float32, device=h_all.device)
    d_gh = torch.empty_like(d_gi)
    with _timed("gru_bwd"):
        _lib.check(_lib.load().rs_gru_bwd(_f32(w_hh).data_ptr(), h_all.data_ptr(), gates.data_ptr(), _p(g_h_all), _p(g_h_last), B, L, H,
                                          d_gi.data_ptr(), d_gh.data_ptr(), _stream()), "rs_gru_bwd")
    _count()
    return d_gi, d_gh


def augru_fwd(gi, att, w_hh, b_hh, want_gates=True):
    """Attention-gated GRU (DIEN's AUGRU): gi (B, L, 3H), att (B, L)  ->  h_all (B, L, H), gates (B, L, 4H) | None."""
    gi, att, w_hh, b_hh = _f32(gi), _f32(att), _f32(w_hh), _f32(b_hh)
    _need_cuda(gi, att, w_hh, b_hh)
    B, L, H3 = gi.shape
    H = H3 // 3
    if tuple(att.shape) != (B, L):
        raise ValueError(f"augru_fwd: att has shape {tuple(att.shape)}, expected {(B, L)}")
    h_all = torch.empty(B, L, H, dtype=torch.float32, device=gi.device)
    gates = torch.empty(B, L, 4 * H, dtype=torch.float32, device=gi.device) if want_gates else None
    if B == 0:
        return h_all, gates
    with _timed("augru_fwd"):
        _lib.check(_lib.load().rs_augru_fwd(gi.data_ptr(), att.data_ptr(), B, L, H, w_hh.data_ptr(), b_hh.data_ptr(), h_all.data_ptr(),
                                            _p(gates), _stream()), "rs_augru_fwd")
    _count()
    return h_all, gates


def augru_bwd(w_hh, att, h_all, gates, g_h_all=None, g_h_last=None):
    """-> d_gi, d_gh (B, L, 3H), d_att (B, L)."""
    B, L, H = h_all.shape
    att, g_h_all, g_h_last = _f32(att), _f32(g_h_all), _f32(g_h_last)
    d_gi = torch.empty(B, L, 3 * H, dtype=torch.float32, device=h_all.device)
    d_gh = torch.empty_like(d_gi)
    d_att = torch.empty(B, L, dtype=torch.float32, device=h_all.device)
    with _timed("augru_bwd"):
        _lib.check(_lib.load().rs_augru_bwd(_f32(w_hh).data_ptr(), att.data_ptr(), h_all.data_ptr(), gates.data_ptr(), _p(g_h_all),
                                            _p(g_h_last), B, L, H, d_gi.data_ptr(), d_gh.data_ptr(), d_att.data_ptr(), _stream()),
                   "rs_augru_bwd")
    _count()
    return d_gi, d_gh, d_att


def _sample_rows(t, name, D):
    """per-sample stride (elements) of a (B, n, D) float32 CUDA view whose rows are contiguous inside a sample"""
    _need_cuda(t)
    if t.dtype != torch.float32 or t.dim() != 3 or t.shape[2] != D or t.stride(2) != 1 or (t.shape[1] > 1 and t.stride(1) != D):
        raise ValueError(f"{name}: expected a float32 (B, n, {D}) view with contiguous rows, got {t.dtype} {tuple(t.shape)} "
                         f"strides {t.stride()}")
    return t.stride(0)


def dien_aux_fwd(h, pos, neg):
    """DIEN auxiliary loss: h (B, L, D) extractor states, pos / neg (B, L-1, D) next-item / negative rows (strided views are
    read in place) -> loss (0-d, mean over the B (L-1) pairs), sig (B, L-1, 2) = (sigma(x+) - 1, sigma(x-))."""
    B, L, D = h.shape
    sh, sp, sn = _sample_rows(h, "dien_aux_fwd h", D), _sample_rows(pos, "dien_aux_fwd pos", D), _sample_rows(neg, "dien_aux_fwd neg", D)
    if tuple(pos.shape) != (B, L - 1, D) or tuple(neg.shape) != (B, L - 1, D):
        raise ValueError(f"dien_aux_fwd: pos {tuple(pos.shape)} / neg {tuple(neg.shape)}, expected {(B, L - 1, D)}")
    sig = torch.empty(B, L - 1, 2, dtype=torch.float32, device=h.device)
    loss = torch.zeros((), dtype=torch.float32, device=h.device)
    if B == 0:
        return loss, sig
    ws = torch.empty(1024, dtype=torch.float32, device=h.device)
    with _timed("dien_aux_fwd"):
        _lib.check(_lib.load().rs_dien_aux_fwd(h.data_ptr(), sh, pos.data_ptr(), sp, neg.data_ptr(), sn, B, L, D, sig.data_ptr(),
                                               loss.data_ptr(), ws.data_ptr(), _stream()), "rs_dien_aux_fwd")
    _count(2)
    return loss, sig


def dien_aux_bwd(h, pos, neg, sig, g):
    """-> dh (B, L, D) (zero at t = L-1), d_pos, d_neg (B, L-1, D) for an upstream gradient g (device scalar tensor)."""
    B, L, D = h.shape
    sh, sp, sn = _sample_rows(h, "dien_aux_bwd h", D), _sample_rows(pos, "dien_aux_bwd pos", D), _sample_rows(neg, "dien_aux_bwd neg", D)
    sig, g = _f32(sig), _f32(g)
    _need_cuda(sig, g)
    if g.numel() != 1:
        raise ValueError("dien_aux_bwd: g must be a scalar")
    dh = torch.empty(B, L, D, dtype=torch.float32, device=h.device)
    d_pos = torch.empty(B, L - 1, D, dtype=torch.float32, device=h.device)
    d_neg = torch.empty_like(d_pos)
    if B == 0:
        return dh, d_pos, d_neg
    with _timed("dien_aux_bwd"):
        _lib.check(_lib.load().rs_dien_aux_bwd(h.data_ptr(), sh, pos.data_ptr(), sp, neg.data_ptr(), sn, B, L, D, sig.data_ptr(),
                                               g.data_ptr(), dh.data_ptr(), d_pos.data_ptr(), d_neg.data_ptr(), _stream()),
                   "rs_dien_aux_bwd")
    _count()
    return dh, d_pos, d_neg


def dien_negatives(hist, num_items, seed, epoch):
    """Negatives of the DIEN auxiliary loss: (B, L-1) int64, slot (b, t) uniform over [0, num_items) and != hist[b, t+1]
    (rs_sample_negatives' Philox stream, counter (b (L-1) + t, attempt block, epoch)).  epoch: int64 device scalar read by
    the kernel (the caller advances it).  Out-of-range history ids set the status word's bit 0, as a lookup does."""
    hist = _i64(hist)
    _need_cuda(hist, epoch)
    if epoch.dtype != torch.int64 or epoch.numel() != 1:
        raise ValueError("dien_negatives: epoch must be an int64 device scalar")
    B, L = hist.shape
    neg = torch.empty(B, max(L - 1, 0), dtype=torch.int64, device=hist.device)
    if neg.numel():
        with _timed("dien_negatives"):
            _lib.check(_lib.load().rs_dien_negatives(hist.data_ptr(), B, L, int(num_items), seed & (2 ** 64 - 1), epoch.data_ptr(),
                                                     neg.data_ptr(), status_word(hist.device).data_ptr(), _stream()),
                       "rs_dien_negatives")
        _count()
    return neg


def afm_fwd(E, W, b, h, want_attw=True):
    """pooled (B, D), attw (B, P) | None."""
    E, W, b, h = _f32(E), _f32(W), _f32(b), _f32(h).reshape(-1)
    _need_cuda(E, W, b, h)
    B, F, D = E.shape
    A = W.shape[1]
    pooled = torch.empty(B, D, dtype=torch.float32, device=E.device)
    attw = torch.empty(B, F * (F - 1) // 2, dtype=torch.float32, device=E.device) if want_attw else None
    if B == 0:
        return pooled, attw
    with _timed("afm_fwd"):
        _lib.check(_lib.load().rs_afm_fwd(E.data_ptr(), B, F, D, A, W.data_ptr(), b.data_ptr(), h.data_ptr(), pooled.data_ptr(),
                                          _p(attw), _stream()), "rs_afm_fwd")
    _count()
    return pooled, attw


_afm_ws = {}


def afm_bwd(E, W, b, h, attw, g_pooled, impl="auto", return_masks=False):
    """-> dE (B,F,D), dW (D,A), db (A), dh (A)  (per-warp partials added in warp order).
    impl "auto": the tcgen05 kernels of afm_tc.cu when rs_afm_bwd_tc_plan accepts the shape; "cuda_cores": rs_afm_bwd.
    return_masks (tensor-core path, tests): a fifth value, the ReLU masks [z > 0] the chain kernel used, (B, P, A) bool."""
    E, W, b, h, g_pooled = _f32(E), _f32(W), _f32(b), _f32(h).reshape(-1), _f32(g_pooled)
    B, F, D = E.shape
    A = W.shape[1]
    lib = _lib.load()
    parts, nbytes = C.c_int32(0), C.c_size_t(0)
    dE = torch.empty_like(E)
    _lib.check(lib.rs_afm_bwd_tc_plan(B, F, D, A, C.byref(parts), C.byref(nbytes)), "rs_afm_bwd_tc_plan")
    if parts.value > 0 and impl != "cuda_cores":
        # tensor-core backward (large batches): partial sums of U = P^T (ds [z > 0]) and m1 = sum ds [z > 0]
        n = parts.value
        Up = torch.empty(n, D, A, dtype=torch.float32, device=E.device)
        m1p = torch.empty(n, A, dtype=torch.float32, device=E.device)
        # the workspace (ds, mask bits, dP: 3.1 GB at C3) is cached per device instead of being allocated every backward.
        # A CUDA-graph capture gets a workspace of its own from the graph's private pool: a cached block is dropped when a
        # larger shape arrives and handed to other tensors, which the replays would then overwrite.
        if torch.cuda.is_current_stream_capturing():
            ws = torch.empty(nbytes.value, dtype=torch.uint8, device=E.device)
        else:
            ws = _afm_ws.get(E.device)
            if ws is None or ws.numel() < nbytes.value:
                _afm_ws[E.device] = None
                ws = _afm_ws[E.device] = torch.empty(nbytes.value, dtype=torch.uint8, device=E.device)
        with _timed("afm_bwd_tc"):
            _lib.check(lib.rs_afm_bwd_tc(E.data_ptr(), B, F, D, A, W.data_ptr(), b.data_ptr(), h.data_ptr(), attw.data_ptr(),
                                         g_pooled.data_ptr(), dE.data_ptr(), Up.data_ptr(), m1p.data_ptr(), n, ws.data_ptr(),
                                         nbytes.value, _stream()), "rs_afm_bwd_tc")
        _count(3)
        U, m1 = Up.sum(dim=0), m1p.sum(dim=0)
        out = (dE, U * h, h * m1, (W * U).sum(dim=0) + b * m1)
        if return_masks:
            NP, AW = F * (F - 1) // 2, A // 32
            off = (B * NP * 4 + 255) // 256 * 256                     # ws layout of rs_afm_bwd_tc: ds | mask bits | dP
            bits = ws[off:off + B * NP * AW * 4].view(torch.int32).view(B, NP, AW, 1)
            masks = ((bits >> torch.arange(32, device=E.device, dtype=torch.int32)) & 1).bool().view(B, NP, A)
            out += (masks,)
        return out
    _lib.check(lib.rs_afm_num_parts(B, F, D, A, C.byref(parts)), "rs_afm_num_parts")
    n = parts.value
    dWp = torch.empty(n, D, A, dtype=torch.float32, device=E.device)
    dbp = torch.empty(n, A, dtype=torch.float32, device=E.device)
    dhp = torch.empty(n, A, dtype=torch.float32, device=E.device)
    with _timed("afm_bwd"):
        _lib.check(lib.rs_afm_bwd(E.data_ptr(), B, F, D, A, W.data_ptr(), b.data_ptr(), h.data_ptr(), attw.data_ptr(),
                                  g_pooled.data_ptr(), dE.data_ptr(), dWp.data_ptr(), dbp.data_ptr(), dhp.data_ptr(), n, _stream()),
                   "rs_afm_bwd")
    _count()
    return dE, dWp.sum(dim=0), dbp.sum(dim=0), dhp.sum(dim=0)


def _din_weights(ws):
    W0, b0, W1, b1, W2, b2 = [_f32(t) for t in ws]
    _need_cuda(W0, b0, W1, b1, W2, b2)
    w = _lib.rs_din_weights()
    w.W0, w.b0, w.W1, w.b1, w.W2, w.b2 = (t.data_ptr() for t in (W0, b0, W1, b1, W2, b2))
    w.H1, w.H2 = W0.shape[0], W1.shape[0]
    return w, (W0, b0, W1, b1, W2, b2)


DIN_TC_MIN_ROWS = 128 * 64     # below this many (b, l) rows the tensor-core tiles cannot fill the machine


def din_tc_supported(D, H1, H2):
    return D in (16, 32, 64) and H1 in (64, 128) and H2 in (32, 64)


DIN_WEIGHTS = "weights"        # `pool` value of din_fwd / din_bwd / din_bwd_tc: the softmax weights (B, L) are the output


def _din_mode(pool):
    """the rs_din_* `pool` argument: RS_DIN_WEIGHTS (2) for DIN_WEIGHTS, else RS_DIN_POOL (1) / RS_DIN_SCALE (0) by truth"""
    return 2 if isinstance(pool, str) and pool == DIN_WEIGHTS else int(bool(pool))


def din_fwd(rows, ws, pool, want_attw=False, impl="auto", want_stash=False):
    """rows (B, L+1, D) = [history | target]; ws = (W0, b0, W1, b1, W2, b2) -> out (B,D) | (B,L,D), attw (B,L) | None.
    pool: true -> (B, D) weighted sum, false -> (B, L, D) scaled history, DIN_WEIGHTS -> (B, L) softmax weights (then
    attw, when wanted, is that same tensor).

    impl: "tc" = hidden layers on the tcgen05 tensor cores (rs_din_fwd_tc), "fused" = the CUDA-core kernel
    (rs_din_fwd), "auto" = tc when the shape is built and there are enough rows to fill the SMs (RS_DIN_TC=0 forces
    fused).  want_stash (training): a third value is returned -- (attw, act0 (B*L, H1), act1 (B*L, H2)), the forward
    activations din_bwd_tc consumes -- or None when the fused kernel ran (its backward recomputes)."""
    rows = _f32(rows)
    _need_cuda(rows)
    B, L1, D = rows.shape
    L = L1 - 1
    w, keep = _din_weights(ws)
    mode = _din_mode(pool)
    out = torch.empty((B, L) if mode == 2 else (B, D) if mode else (B, L, D), dtype=torch.float32, device=rows.device)
    if impl == "auto":
        fused_ok = D in (16, 32, 64) and (w.H1, w.H2) in ((128, 64), (64, 32))
        big = B * L >= DIN_TC_MIN_ROWS and os.environ.get("RS_DIN_TC", "1") != "0"
        impl = "tc" if din_tc_supported(D, w.H1, w.H2) and (big or not fused_ok) else "fused"
    stash_tc = want_stash and impl == "tc"
    if mode == 2:
        attw = out if (want_attw or stash_tc) else None
    else:
        attw = torch.empty(B, L, dtype=torch.float32, device=rows.device) if (want_attw or stash_tc) else None
    kattw = None if mode == 2 else attw      # the weights mode writes its weights to `out` only
    if B == 0:
        return (out, attw, None) if want_stash else (out, attw)
    lib = _lib.load()
    if impl == "tc":
        nbytes = C.c_size_t(0)
        _lib.check(lib.rs_din_fwd_tc_ws_bytes(B, L, D, w.H1, w.H2, C.byref(nbytes)), "rs_din_fwd_tc_ws_bytes")
        scratch = torch.empty(nbytes.value, dtype=torch.uint8, device=rows.device)
        act0 = torch.empty(B * L, w.H1, dtype=torch.float32, device=rows.device) if stash_tc else None
        act1 = torch.empty(B * L, w.H2, dtype=torch.float32, device=rows.device) if stash_tc else None
        with _timed("din_fwd_tc"):
            _lib.check(lib.rs_din_fwd_tc(rows.data_ptr(), B, L, D, C.byref(w), mode, out.data_ptr(), _p(kattw), _p(act0),
                                         _p(act1), scratch.data_ptr(), nbytes.value, _stream()), "rs_din_fwd_tc")
        _count(3)
        return (out, attw, (attw, act0, act1) if stash_tc else None) if want_stash else (out, attw)
    with _timed("din_fwd"):
        _lib.check(lib.rs_din_fwd(rows.data_ptr(), B, L, D, C.byref(w), mode, out.data_ptr(), _p(kattw), _stream()),
                   "rs_din_fwd")
    _count()
    return (out, attw, None) if want_stash else (out, attw)


def din_bwd_tc(rows, ws, pool, g_out, stash):
    """Backward of the tensor-core forward from its stash -> d_rows (B, L+1, D), (dW0, db0, dW1, db1, dW2, db2).
    rs_din_bwd_tc runs the data-gradient chain (two fused tcgen05 GEMMs per 128-row tile); the weight gradients are
    reductions over all B*L rows: two rs_gemm_tn_3xtf32 calls plus small sums / products on the per-sample terms."""
    rows, g_out = _f32(rows), _f32(g_out)
    attw, act0, act1 = stash
    B, L1, D = rows.shape
    L = L1 - 1
    w, keep = _din_weights(ws)
    W0 = keep[0]
    H1, H2 = w.H1, w.H2
    dev = rows.device
    d_rows = torch.empty_like(rows)
    dz0 = torch.empty(B, L1, H1, dtype=torch.float32, device=dev)
    dz1 = torch.empty(B * L, H2, dtype=torch.float32, device=dev)
    ds = torch.empty(B, L, dtype=torch.float32, device=dev)
    with _timed("din_bwd_tc"):
        _lib.check(_lib.load().rs_din_bwd_tc(rows.data_ptr(), B, L, D, C.byref(w), _din_mode(pool), g_out.data_ptr(), attw.data_ptr(),
                                             act0.data_ptr(), act1.data_ptr(), d_rows.data_ptr(), dz0.data_ptr(), dz1.data_ptr(),
                                             ds.data_ptr(), _stream()), "rs_din_bwd_tc")
    _count(2)
    with _timed("din_bwd_tc_weights"):
        dW1 = gemm_tn(act0, dz1).t().contiguous()                    # (H2, H1)
        dWab = gemm_tn(dz0.view(B * L1, H1), rows.view(B * L1, D))   # (H1, D): the target slots of dz0 are zero
        db1 = dz1.sum(0)
        dW2 = ds.view(1, B * L) @ act1                               # (1, H2)
        db2 = ds.sum().view(1)
        dtb = dz0.sum(1)                                             # (B, H1): gradient of the per-sample target term
        t = rows[:, L]
        dWt = dtb.t() @ t                                            # (H1, D)
        d_rows[:, L] = dtb @ (W0[:, 2 * D:] - W0[:, D:2 * D])
        dW0 = torch.cat([dWab, dWab - dWt, dWt], dim=1)
    return d_rows, (dW0, dtb.sum(0), dW1, db1, dW2, db2)


def din_bwd(rows, ws, pool, g_out):
    """-> d_rows (B, L+1, D), (dW0, db0, dW1, db1, dW2, db2)."""
    rows, g_out = _f32(rows), _f32(g_out)
    B, L1, D = rows.shape
    L = L1 - 1
    w, keep = _din_weights(ws)
    H1, H2 = w.H1, w.H2
    lib = _lib.load()
    parts = C.c_int32(0)
    _lib.check(lib.rs_din_num_parts(B, C.byref(parts)), "rs_din_num_parts")
    n, dev = parts.value, rows.device
    d_rows = torch.empty_like(rows)
    mk = lambda *shape: torch.empty(n, *shape, dtype=torch.float32, device=dev)   # noqa: E731
    dWab, dWt, dW1, db0, db1, dW2, db2 = mk(H1, D), mk(H1, D), mk(H2, H1), mk(H1), mk(H2), mk(H2), mk()
    with _timed("din_bwd"):
        _lib.check(lib.rs_din_bwd(rows.data_ptr(), B, L, D, C.byref(w), _din_mode(pool), g_out.data_ptr(), d_rows.data_ptr(),
                                  dWab.data_ptr(), dWt.data_ptr(), dW1.data_ptr(), db0.data_ptr(), db1.data_ptr(), dW2.data_ptr(),
                                  db2.data_ptr(), n, _stream()), "rs_din_bwd")
    _count()
    dWab, dWt = dWab.sum(0), dWt.sum(0)
    dW0 = torch.cat([dWab, dWab - dWt, dWt], dim=1)
    return d_rows, (dW0, db0.sum(0), dW1.sum(0), db1.sum(0), dW2.sum(0).view(1, H2), db2.sum(0).view(1))


def gemm_tn(A, B):
    """A^T B for row-major A (K, M), B (K, N) on tcgen05 (3xTF32, fp32 accumulate in TMEM).  M <= 128, N <= 256."""
    A, B = _f32(A), _f32(B)
    _need_cuda(A, B)
    K, M = A.shape
    N = B.shape[1]
    lib = _lib.load()
    nbytes = C.c_size_t(0)
    _lib.check(lib.rs_gemm_tn_ws_bytes(K, M, N, C.byref(nbytes)), "rs_gemm_tn_ws_bytes")
    ws = torch.empty(nbytes.value // 4 + 1, dtype=torch.float32, device=A.device)
    out = torch.empty(M, N, dtype=torch.float32, device=A.device)
    with _timed("gemm_tn_3xtf32"):
        _lib.check(lib.rs_gemm_tn_3xtf32(A.data_ptr(), B.data_ptr(), K, M, N, out.data_ptr(), ws.data_ptr(), nbytes.value, _stream()),
                   "rs_gemm_tn_3xtf32")
    _count(2)
    return out


def gemm_nt(A, W, bias=None, rowbias=None, rb_group=1, relu=False, mask=None, M=None, a_rows=None):
    """epilogue(A W^T) on tcgen05 (3xTF32).  A (M, K) contiguous, or -- with a_rows=(group, group_stride, lda) -- a
    strided view whose row r lives at A.data_ptr + (r // group)*group_stride + (r % group)*lda floats.
    W (N, K) torch Linear layout.  Epilogue: + bias[n] + rowbias[r // rb_group][n], ReLU, zero where mask <= 0."""
    W = _f32(W)
    _need_cuda(A, W)
    g = _lib.rs_gemm_nt()
    N, K = W.shape
    if a_rows is None:
        A = _f32(A)
        M = A.shape[0]
        g.lda, g.a_group, g.a_group_stride = A.shape[1], 0, 0
    else:
        g.a_group, g.a_group_stride, g.lda = a_rows
    out = torch.empty(M, N, dtype=torch.float32, device=W.device)
    g.A, g.B, g.C = A.data_ptr(), W.data_ptr(), out.data_ptr()
    bias, rowbias, mask = _f32(bias), _f32(rowbias), _f32(mask)
    g.bias, g.rowbias, g.mask = _p(bias), _p(rowbias), _p(mask)
    g.M, g.ldb, g.rb_group, g.ldm, g.ldc = M, K, rb_group, N, N
    g.K, g.N, g.relu = K, N, int(bool(relu))
    with _timed(f"gemm_nt[{N}x{K}]"):
        _lib.check(_lib.load().rs_gemm_nt_3xtf32(C.byref(g), _stream()), "rs_gemm_nt_3xtf32")
    _count()
    return out


def _rank_status(st, k, who):
    v = int(st.item())
    if v & 2:
        raise RuntimeError(f"{who}: selected index k={k} out of range (a segment is shorter than k)")
    if v & 4:
        raise RuntimeError(f"{who}: a segment is longer than the max_len it was launched with")


def rank_segments(scores, k, seg_start=None, seg_len=None, max_len=None, values=False, check=True):
    """Per-segment descending top-k positions (k == segment length: the full ranking) -- one launch for all users.

    scores: flat fp32; segments either uniform (``seg_len``) or given by ``seg_start`` (int64, S+1 offsets; pass
    ``max_len`` = an upper bound of the segment lengths).  Returns idx (S, k) int64 positions inside each segment
    [, val (S, k)].  Ties rank the lower position first.  ``check`` reads the status word (one sync)."""
    scores = _f32(scores).view(-1)
    _need_cuda(scores, seg_start)
    if seg_start is None:
        if seg_len is None or seg_len <= 0 or scores.numel() % seg_len:
            raise ValueError("rank_segments: uniform segments need seg_len dividing scores.numel()")
        S, max_len, ss = scores.numel() // seg_len, seg_len, None
    else:
        ss = _i64(seg_start)
        S = ss.numel() - 1
        if max_len is None:
            max_len = int((ss[1:] - ss[:-1]).max().item()) if S > 0 else 1
    idx = torch.empty(S, k, dtype=torch.int64, device=scores.device)
    val = torch.empty(S, k, dtype=torch.float32, device=scores.device) if values else None
    if S > 0:
        st = torch.zeros(1, dtype=torch.int32, device=scores.device)
        with _timed("rank_segments"):
            _lib.check(_lib.load().rs_rank_segments(scores.data_ptr(), _p(ss), S, max(int(max_len), 1), k, idx.data_ptr(), _p(val),
                                                    st.data_ptr(), _stream()), "rs_rank_segments")
        _count()
        if check:
            _rank_status(st, k, "rank_segments")
    return (idx, val) if values else idx


def mf_rank(user_rows, item_rows, k, values=False, check=True):
    """Fused ``topk(user_rows @ item_rows.T, k, dim=1)``: the (users, items) score matrix never reaches HBM."""
    U, V = _f32(user_rows), _f32(item_rows)
    _need_cuda(U, V)
    if U.dim() != 2 or V.dim() != 2 or U.shape[1] != V.shape[1]:
        raise ValueError("mf_rank: user_rows (U, W) and item_rows (I, W) must share W")
    nu, ni = U.shape[0], V.shape[0]
    if k > ni:
        raise RuntimeError(f"mf_rank: selected index k={k} out of range ({ni} items)")
    idx = torch.empty(nu, k, dtype=torch.int64, device=U.device)
    val = torch.empty(nu, k, dtype=torch.float32, device=U.device) if values else None
    if nu > 0:
        st = torch.zeros(1, dtype=torch.int32, device=U.device)
        lib, nbytes = _lib.load(), C.c_size_t(0)
        _lib.check(lib.rs_mf_rank_ws_bytes(nu, ni, U.shape[1], k, C.byref(nbytes)), "rs_mf_rank_ws_bytes")
        ws = torch.empty(nbytes.value, dtype=torch.uint8, device=U.device) if nbytes.value else None
        with _timed("mf_rank"):
            _lib.check(lib.rs_mf_rank(U.data_ptr(), V.data_ptr(), nu, ni, U.shape[1], k, idx.data_ptr(), _p(val), st.data_ptr(),
                                      _p(ws), nbytes.value, _stream()), "rs_mf_rank")
        _count(2 if ws is not None else 1)
        if check:
            _rank_status(st, k, "mf_rank")
    return (idx, val) if values else idx


def sample_negatives(excluded_keys, num_user, num_item, num_negatives, seed, epoch=0):
    """OPTIONAL device sampler (not the reference's python-`random` stream; see include/recsys_b200.h).
    excluded_keys: ascending int64 CUDA tensor of user * num_item + item.  -> (users, items) int64, user-major."""
    keys = _i64(excluded_keys).view(-1)
    _need_cuda(keys)
    total = num_user * num_negatives
    users = torch.empty(total, dtype=torch.int64, device=keys.device)
    items = torch.empty(total, dtype=torch.int64, device=keys.device)
    if total:
        st = torch.zeros(1, dtype=torch.int32, device=keys.device)
        with _timed("sample_negatives"):
            _lib.check(_lib.load().rs_sample_negatives(keys.data_ptr() if keys.numel() else None, keys.numel(), num_user, num_item,
                                                       num_negatives, seed & (2 ** 64 - 1), epoch, users.data_ptr(), items.data_ptr(),
                                                       st.data_ptr(), _stream()), "rs_sample_negatives")
        _count()
        if int(st.item()) & 8:
            raise RuntimeError("sample_negatives: a user has (almost) every item observed; no free item found")
    return users, items


def assemble_features(users, items, user_feat, item_feat):
    """(B, 2 + FU + FI) fp32 rows [user, item, user_feat[user], item_feat[item]] -- data/reader.py:98-101 on the device."""
    users, items = _i64(users).view(-1), _i64(items).view(-1)
    user_feat, item_feat = _f32(user_feat), _f32(item_feat)
    _need_cuda(users, items, user_feat, item_feat)
    B, FU, FI = users.numel(), user_feat.shape[1], item_feat.shape[1]
    out = torch.empty(B, 2 + FU + FI, dtype=torch.float32, device=users.device)
    if B:
        with _timed("assemble_features"):
            _lib.check(_lib.load().rs_assemble_features(users.data_ptr(), items.data_ptr(), user_feat.data_ptr(), user_feat.shape[0], FU,
                                                        item_feat.data_ptr(), item_feat.shape[0], FI, B, out.data_ptr(),
                                                        status_word(users.device).data_ptr(), _stream()), "rs_assemble_features")
        _count()
    return out
