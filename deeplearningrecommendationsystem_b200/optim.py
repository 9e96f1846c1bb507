"""Optimizer protocol seen by Trainer (reference trainer/trainer.py:25,39: ``zero_grad()`` + ``step()``).

``FusedRowOptimizer`` owns the update of every embedding table that runs in *fused sparse* mode: backward only
stashes (ids, Jacobian rows, upstream scalars); ``step()`` runs the deterministic sort / segment-reduce fused with
the SGD / lazy-Adam row update (rs_dedup_sort + rs_segment_update) and then delegates all dense parameters to a
stock torch optimizer.  Tables in this mode have ``requires_grad=False`` so nothing is applied twice.

Semantics: SGD here equals the reference's dense SGD exactly (untouched rows have zero gradient).  Row-wise
(lazy) Adam differs from the reference's dense ``optim.Adam(weight_decay=...)`` for untouched rows by design; use
the default dense-gradient mode of the drop-in modules + ``torch.optim.Adam`` (or ``DenseAdam`` below) when the
reference's exact Adam trajectory is required.
"""
import torch

from . import ops


class FusedRowOptimizer:
    """One ``step()`` is one optimizer step per table, also when the model ran several forwards since ``zero_grad()``.
    With ``kind="adam"`` or ``weight_decay != 0`` the pending lookups of a table are merged and updated once on their
    summed gradient, as ``torch.optim`` steps once on the accumulated ``.grad``: the moments advance once and the decay
    term is applied once.  Plain SGD without decay applies the forwards one after another (the same result up to
    rounding).  A row-sharded table takes one forward per step with Adam or weight decay (several raise), and so does
    the stash-free FFM forward (``RS_FFM_RECOMPUTE=1``) with weight decay.

    Multi-GPU: row-sharded tables are stepped by their owners; the replicated small tables of the hybrid placement are
    stepped by rs_replica_update, which updates only rows some rank's batch touched (lazy, as on one GPU) and keeps each
    rank's slice of the Adam moments (``adam_m_small`` / ``adam_v_small``, bounds ``small_slice``).  Plain SGD without
    decay there steps every element with rs_replica_sgd (an untouched row's gradient is zero)."""

    def __init__(self, model, dense_optimizer=None, lr=0.01, kind="sgd", weight_decay=0.0, betas=(0.9, 0.999), eps=1e-8,
                 data_parallel=True):
        """data_parallel: average the dense parameters' gradients over the process group before the dense step (the
        replicated-parameter half of the multi-GPU partition); False for a model that lives on one rank only."""
        if kind not in ("sgd", "adam"):
            raise ValueError("kind must be 'sgd' or 'adam'")
        self.model, self.dense = model, dense_optimizer
        self.lr, self.kind, self.weight_decay, self.betas, self.eps = lr, kind, weight_decay, betas, eps
        self.step_count = 0
        self.data_parallel = data_parallel
        for m in self._sparse_modules():
            if hasattr(m, "bind_row_optimizer"):
                m.bind_row_optimizer(self)

    def _sparse_modules(self):
        return [m for m in self.model.modules() if hasattr(m, "apply_pending")]

    def zero_grad(self, set_to_none=True):
        if self.dense is not None:
            self.dense.zero_grad(set_to_none=set_to_none)
        for m in self._sparse_modules():
            m.clear_pending()

    def step(self):
        self.step_count += 1
        for m in self._sparse_modules():
            m.apply_pending(self)
        if self.dense is not None and not self.data_parallel:
            self.dense.step()
        elif self.dense is not None:
            from .dist import allreduce_dense_grads
            fabric = next((m.exchange.fabric for m in self._sparse_modules()
                           if getattr(m, "exchange", None) is not None and hasattr(m.exchange, "fabric")), None)
            allreduce_dense_grads([p for g in self.dense.param_groups for p in g["params"]], fabric=fabric)
            self.dense.step()


class DenseAdam(torch.optim.Optimizer):
    """torch.optim.Adam's arithmetic (L2 weight decay folded into the gradient, every element moves every step;
    reference scripts/deepfm.py:55) as ONE fused kernel per parameter (rs_adam_dense)."""

    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0):
        super().__init__(params, dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay))

    @torch.no_grad()
    def step(self, closure=None):
        for group in self.param_groups:
            for p in group["params"]:
                if p.grad is None:
                    continue
                st = self.state[p]
                if not st:
                    st["step"] = 0
                    st["exp_avg"] = torch.zeros_like(p, memory_format=torch.contiguous_format)
                    st["exp_avg_sq"] = torch.zeros_like(p, memory_format=torch.contiguous_format)
                st["step"] += 1
                if not p.is_contiguous():
                    raise RuntimeError("DenseAdam needs contiguous parameters")
                ops.adam_dense(p.data, p.grad.contiguous(), st["exp_avg"], st["exp_avg_sq"], st["step"], lr=group["lr"],
                               wd=group["weight_decay"], betas=group["betas"], eps=group["eps"])
