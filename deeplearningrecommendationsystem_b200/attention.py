"""Attention pooling (AFM), target attention (DIN / DIEN), the GRU / AUGRU recurrences and DIEN's auxiliary loss of the
drop-in modules."""
import torch


class _AFMPool(torch.autograd.Function):
    """rs_afm_fwd / rs_afm_bwd: the pair tensor stays in shared memory, parameter gradients are fixed-order sums."""

    @staticmethod
    def forward(ctx, E, W, b, h):
        from . import ops
        need = any(t.requires_grad for t in (E, W, b, h))
        pooled, attw = ops.afm_fwd(E, W.detach(), b.detach(), h.detach(), want_attw=need)
        if need:
            ctx.save_for_backward(E, W, b, h, attw)
        return pooled

    @staticmethod
    def backward(ctx, g):
        from . import ops
        E, W, b, h, attw = ctx.saved_tensors
        dE, dW, db, dh = ops.afm_bwd(E, W.detach(), b.detach(), h.detach(), attw, g.contiguous())
        return dE, dW, db, dh.view_as(h)


def afm_pool(E, W, b, h):
    """Attention pooling over the pairwise Hadamard products of E (B, F, D) -> (B, D)   reference model/afm.py:55-65."""
    return _AFMPool.apply(E.contiguous(), W, b, h)


class _DINAttention(torch.autograd.Function):
    """rs_din_fwd / rs_din_bwd on rows (B, L+1, D) = [history | target].  Large batches run the hidden layers on the
    tensor cores (rs_din_fwd_tc); that forward stashes its ReLU outputs and rs_din_bwd_tc consumes them, while the
    CUDA-core kernel pair recomputes instead."""

    @staticmethod
    def forward(ctx, rows, pool, W0, b0, W1, b1, W2, b2):
        from . import ops
        ws = (W0, b0, W1, b1, W2, b2)
        need = any(ctx.needs_input_grad)
        out, _, stash = ops.din_fwd(rows, [t.detach() for t in ws], pool, want_stash=need)
        ctx.pool, ctx.tc = pool, stash is not None
        ctx.save_for_backward(rows, *ws, *(stash or ()))
        return out

    @staticmethod
    def backward(ctx, g):
        from . import ops
        rows, *rest = ctx.saved_tensors
        ws, stash = rest[:6], rest[6:]
        if ctx.tc:
            d_rows, dws = ops.din_bwd_tc(rows, [t.detach() for t in ws], ctx.pool, g.contiguous(), stash)
        else:
            d_rows, dws = ops.din_bwd(rows, [t.detach() for t in ws], ctx.pool, g.contiguous())
        return (d_rows, None, *dws)


def din_attention(rows, unit, pool):
    """softmax_L(MLP([h, h-t, t])) applied to the history                               reference model/din.py:39-47.
    rows (B, L+1, D): gathered history rows followed by the target row; unit = Sequential(Linear, ReLU, Linear, ReLU,
    Linear).  pool=True -> (B, D) weighted sum; pool=False -> (B, L, D) scaled history (model/dien.py:33-37).
    rs_din_fwd / rs_din_bwd: for B*L >= 8192 rows the tcgen05 kernels of din_tc.cu (both hidden layers fused per
    128-row tile, 3xTF32), otherwise the CUDA-core kernel pair (ops.din_fwd picks)."""
    l0, l1, l2 = unit[0], unit[2], unit[4]
    return _DINAttention.apply(rows.contiguous(), pool, l0.weight, l0.bias, l1.weight, l1.bias, l2.weight, l2.bias)


def din_attention_weights(rows, unit):
    """The softmax weights w (B, L) of din_attention themselves (the DIEN paper's attention scores), bit-identical to the
    weights the pooling and scaling modes apply; the gradient with respect to w flows back through the unit into rows."""
    from . import ops
    return din_attention(rows, unit, ops.DIN_WEIGHTS)


class _GRURecurrence(torch.autograd.Function):
    """L sequential GRU steps on precomputed input projections (rs_gru_fwd / rs_gru_bwd).  Returns h_L (B, H)."""

    @staticmethod
    def forward(ctx, gi, w_hh, b_hh):
        from . import ops
        need = gi.requires_grad or w_hh.requires_grad or b_hh.requires_grad
        h_all, gates = ops.gru_fwd(gi, w_hh.detach(), b_hh.detach(), want_gates=need)
        if need:
            ctx.save_for_backward(w_hh, h_all, gates)
        return h_all[:, -1].clone()

    @staticmethod
    def backward(ctx, g_last):
        from . import ops
        w_hh, h_all, gates = ctx.saved_tensors
        B, L, H = h_all.shape
        d_gi, d_gh = ops.gru_bwd(w_hh.detach(), h_all, gates, g_h_last=g_last.contiguous())
        h_prev = torch.cat([torch.zeros(B, 1, H, device=h_all.device), h_all[:, :-1]], dim=1)
        flat = d_gh.view(B * L, 3 * H)
        return d_gi, flat.t() @ h_prev.reshape(B * L, H), flat.sum(dim=0)


class _GRUSequence(torch.autograd.Function):
    """_GRURecurrence returning every h_t (B, L, H); the backward runs rs_gru_bwd from the per-step gradient g_h_all."""

    @staticmethod
    def forward(ctx, gi, w_hh, b_hh):
        from . import ops
        need = any(ctx.needs_input_grad)
        h_all, gates = ops.gru_fwd(gi, w_hh.detach(), b_hh.detach(), want_gates=need)
        if need:
            ctx.save_for_backward(w_hh, h_all, gates)
        return h_all

    @staticmethod
    def backward(ctx, g_all):
        from . import ops
        w_hh, h_all, gates = ctx.saved_tensors
        B, L, H = h_all.shape
        d_gi, d_gh = ops.gru_bwd(w_hh.detach(), h_all, gates, g_h_all=g_all.contiguous())
        h_prev = torch.cat([torch.zeros(B, 1, H, device=h_all.device), h_all[:, :-1]], dim=1)
        flat = d_gh.view(B * L, 3 * H)
        return d_gi, flat.t() @ h_prev.reshape(B * L, H), flat.sum(dim=0)


def _check_gru(gru, name):
    if gru.num_layers != 1 or gru.bidirectional or not gru.batch_first or gru.hidden_size not in (8, 16, 32, 64):
        raise NotImplementedError(f"{name}: single-layer batch_first GRU with hidden size in {{8,16,32,64}}")


def gru_last_hidden(x, gru):
    """hidden[-1] of a single-layer batch_first GRU started from zeros                  reference model/dien.py:61-64.
    Input projection = one library GEMM; the recurrence and its BPTT run in the hand-written kernels."""
    _check_gru(gru, "gru_last_hidden")
    gi = torch.nn.functional.linear(x, gru.weight_ih_l0, gru.bias_ih_l0)
    return _GRURecurrence.apply(gi, gru.weight_hh_l0, gru.bias_hh_l0)


def gru_sequence(x, gru):
    """Every hidden state (B, L, H) of a single-layer batch_first GRU started from zeros (nn.GRU's `output`): the DIEN
    paper's interest extractor.  Same kernels as gru_last_hidden; the backward takes a gradient for every h_t."""
    _check_gru(gru, "gru_sequence")
    gi = torch.nn.functional.linear(x, gru.weight_ih_l0, gru.bias_ih_l0)
    return _GRUSequence.apply(gi, gru.weight_hh_l0, gru.bias_hh_l0)


class _DIENAux(torch.autograd.Function):
    """rs_dien_aux_fwd / rs_dien_aux_bwd; the upstream gradient stays on the device."""

    @staticmethod
    def forward(ctx, h, pos, neg):
        from . import ops
        loss, sig = ops.dien_aux_fwd(h, pos, neg)
        ctx.save_for_backward(h, pos, neg, sig)
        return loss

    @staticmethod
    def backward(ctx, g):
        from . import ops
        h, pos, neg, sig = ctx.saved_tensors
        return ops.dien_aux_bwd(h, pos, neg, sig, g.reshape(1))


def dien_aux_loss(h, pos, neg):
    """The DIEN paper's auxiliary loss (eq. 5, inner-product form), the mean over the B (L-1) pairs (b, t < L-1) of
    softplus(-<h_t, pos_t>) + softplus(<h_t, neg_t>): h (B, L, D) extractor states, pos (B, L-1, D) the embeddings of the
    next clicked items e_{t+1}, neg (B, L-1, D) those of drawn negatives.  Strided views (slices of one lookup) are read
    in place.  D in {16, 32, 64}."""
    return _DIENAux.apply(h, pos, neg)


class _AUGRURecurrence(torch.autograd.Function):
    """L sequential AUGRU steps on precomputed input projections (rs_augru_fwd / rs_augru_bwd).  Returns h_L (B, H)."""

    @staticmethod
    def forward(ctx, gi, att, w_hh, b_hh):
        from . import ops
        need = any(ctx.needs_input_grad)
        h_all, gates = ops.augru_fwd(gi, att, w_hh.detach(), b_hh.detach(), want_gates=need)
        if need:
            ctx.save_for_backward(att, w_hh, h_all, gates)
        return h_all[:, -1].clone()

    @staticmethod
    def backward(ctx, g_last):
        from . import ops
        att, w_hh, h_all, gates = ctx.saved_tensors
        B, L, H = h_all.shape
        d_gi, d_gh, d_att = ops.augru_bwd(w_hh.detach(), att, h_all, gates, g_h_last=g_last.contiguous())
        h_prev = torch.cat([torch.zeros(B, 1, H, device=h_all.device), h_all[:, :-1]], dim=1)
        flat = d_gh.view(B * L, 3 * H)
        return d_gi, d_att, flat.t() @ h_prev.reshape(B * L, H), flat.sum(dim=0)


def augru_last_hidden(x, att, gru):
    """h_L of the DIEN paper's attention-gated GRU (AUGRU) with the weights of `gru` (an nn.GRU), h0 = 0:
    u = att[:, t] (1 - z),  h_t = (1 - u) h_{t-1} + u n  with torch's gates r, z, n.  x (B, L, D) is NOT scaled by att;
    att (B, L) gates the update instead.  att == 1 gives gru_last_hidden, att == 0 gives zeros.
    Input projection = one library GEMM; the recurrence and its BPTT (including d att) run in the hand-written kernels."""
    _check_gru(gru, "augru_last_hidden")
    if att.dim() != 2 or tuple(att.shape) != tuple(x.shape[:2]):
        raise ValueError(f"augru_last_hidden: att has shape {tuple(att.shape)}, expected {tuple(x.shape[:2])}")
    gi = torch.nn.functional.linear(x, gru.weight_ih_l0, gru.bias_ih_l0)
    return _AUGRURecurrence.apply(gi, att.contiguous(), gru.weight_hh_l0, gru.bias_hh_l0)
