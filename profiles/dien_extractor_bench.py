"""DIEN's interest extractor and auxiliary loss at the C4 shape: B = 8192, L = 100, D = 64, one GPU.

1. Kernels: rs_dien_negatives, rs_dien_aux_fwd and rs_dien_aux_bwd per call, with the algorithmic bytes over time
   against the 7.7 TB/s HBM3e data-sheet figure, beside the same loss composed from torch ops (gather, bmm,
   logsigmoid, autograd) on the same inputs; both losses are printed.
2. The DIEN train step (1 M-row item table, fused sparse rows, SGD lr 0.01, Trainer.train_loop as bench.py --workload c4
   builds it), eager and CUDA-graph replayed (GraphedTrainStep), for evolution="gru", "augru", "augru" + extractor with
   aux_weight = 0 and "augru" + extractor with aux_weight = 1: what each layer of the paper costs.

Times: CUDA events around `--iters` back-to-back calls or steps, repeated `--rounds` times with the variants alternating
inside every round; the median over rounds is printed (and the spread, min..max).  Every variant is warmed up first.
The kernels' operands (0.2 GB each) and the step's working set exceed the 126 MB L2.

    python profiles/dien_extractor_bench.py [--iters 20] [--rounds 7] [--out FILE]
"""
import argparse
import os
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from augru_bench import card, report, run, zipf_ids  # noqa: E402
from deeplearningrecommendationsystem_b200 import attention, ops  # noqa: E402

B, L, D, ITEMS, LR = 8192, 100, 64, 1_000_000, 0.01
HBM = 7.7e12          # bytes/s, NVIDIA's HGX B200 data sheet, one GPU


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--out", default=None, help="also write the report to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a GPU")
    from deeplearningrecommendationsystem_b200 import model as M
    from deeplearningrecommendationsystem_b200.graph import GraphedTrainStep
    from deeplearningrecommendationsystem_b200.optim import FusedRowOptimizer
    from deeplearningrecommendationsystem_b200.trainer import Trainer
    out = []

    def emit(*lines):
        for line in lines:
            print(line, flush=True)
            out.append(line)
    emit(f"card: {card()}", f"shape: B = {B}, L = {L}, D = {D}; {args.rounds} rounds x {args.iters} calls, medians", "")
    g = torch.Generator(device="cuda").manual_seed(0)

    # 1. kernels, on the layout the model hands them: h (B, L, D) contiguous, pos / neg slices of one (B, 2L, D) lookup
    table = torch.randn(ITEMS, D, device="cuda", generator=g) * 0.1
    hist = zipf_ids(ITEMS, (B, L), g)
    epoch = torch.zeros((), dtype=torch.int64, device="cuda")
    neg_ids = ops.dien_negatives(hist, ITEMS, 12345, epoch)
    ids = torch.cat([hist, torch.randint(0, ITEMS, (B, 1), generator=g, device="cuda"), neg_ids], dim=1)
    rows = table[ids]
    h = (torch.randn(B, L, D, device="cuda", generator=g) * 0.3)
    pos, neg = rows[:, 1:L], rows[:, L + 1:]
    one = torch.ones((), device="cuda")
    loss, sig = ops.dien_aux_fwd(h, pos, neg)
    P = B * (L - 1)
    byts = {"rs_dien_negatives": P * 8 * 2,                       # hist[b, t+1] read, neg written
            "rs_dien_aux_fwd": 3 * P * D * 4 + P * 8,               # h_t, e_{t+1}, e^_{t+1} read; (sig0, sig1) written
            "rs_dien_aux_bwd": 3 * P * D * 4 + P * 8 + (B * L + 2 * P) * D * 4}   # + dh, d_pos, d_neg written

    # both routes start from the same leaves -- h and the (B, 2L, D) rows of one lookup -- and end with their gradients
    hr, rows_t = h.clone().requires_grad_(True), rows.clone().requires_grad_(True)
    hr2, rows_r = h.clone().requires_grad_(True), rows.clone().requires_grad_(True)
    sel = torch.arange(L - 1, device="cuda")

    def torch_loss():
        """the same loss from torch ops: index_select of the pairs' rows, bmm for the dot products, logsigmoid, autograd"""
        hp = hr.index_select(1, sel).reshape(P, 1, D)
        xp = torch.bmm(hp, rows_t.index_select(1, sel + 1).reshape(P, D, 1)).view(-1)
        xn = torch.bmm(hp, rows_t.index_select(1, sel + L + 1).reshape(P, D, 1)).view(-1)
        return -(torch.nn.functional.logsigmoid(xp) + torch.nn.functional.logsigmoid(-xn)).mean()

    def torch_fwd_bwd():
        torch_loss().backward()

    def lib_loss_bwd():
        attention.dien_aux_loss(hr2, rows_r[:, 1:L], rows_r[:, L + 1:]).backward()
    t = run({"rs_dien_negatives": lambda: ops.dien_negatives(hist, ITEMS, 12345, epoch),
             "rs_dien_aux_fwd": lambda: ops.dien_aux_fwd(h, pos, neg),
             "rs_dien_aux_bwd": lambda: ops.dien_aux_bwd(h, pos, neg, sig, one)}, args.iters * 5, args.rounds)
    emit("1. auxiliary-loss kernels, per call (algorithmic bytes / median time; data sheet 7.7 TB/s)")
    for k, v in t.items():
        med = v[len(v) // 2] * 1e-3
        emit(f"  {k:40s} {med * 1e6:9.1f} us  (min {v[0] * 1e3:.1f}, max {v[-1] * 1e3:.1f})  {byts[k] / 1e9:.3f} GB  "
             f"{byts[k] / med / 1e12:.2f} TB/s = {byts[k] / med / HBM:.2f} of 7.7 TB/s")
    with torch.no_grad():
        lt = torch_loss()
    emit(f"  loss: kernels {float(loss):.7f}, torch ops {float(lt):.7f}, |diff| {abs(float(loss) - float(lt)):.2e}")
    t = run({"kernels: dien_aux_loss fwd + bwd": lib_loss_bwd,
             "torch ops: index_select + bmm + logsigmoid": torch_fwd_bwd}, args.iters, args.rounds)
    emit(*report("  forward + backward from (h, rows) to their gradients through autograd, per call", t, "ms", 1.0,
                 "kernels: dien_aux_loss fwd + bwd"))
    del rows, rows_r, rows_t, h, hr, hr2, table, sig, pos, neg, ids
    torch.cuda.empty_cache()
    emit("")

    # 2. the DIEN train step
    pool = []
    for _ in range(4):
        hh = zipf_ids(ITEMS, (B, L), g)
        tgt = torch.randint(0, ITEMS, (B,), generator=g, device="cuda")
        pool.append(((hh, tgt), (torch.rand(B, 1, generator=g, device="cuda") < 0.3).float()))
    variants = {"gru": dict(evolution="gru"), "augru": dict(evolution="augru"),
                "augru + extractor, aux_weight=0": dict(evolution="augru", extractor=True, aux_weight=0.0),
                "augru + extractor, aux_weight=1": dict(evolution="augru", extractor=True, aux_weight=1.0)}
    steps = {}

    def build(kw):
        torch.manual_seed(0)
        m = M.DIEN(ITEMS, D, **kw).cuda().fuse_embedding_updates()
        return m, FusedRowOptimizer(m, torch.optim.SGD([p for p in m.parameters() if p.requires_grad], lr=LR), lr=LR)
    for name, kw in variants.items():
        # one model per leg: the eager and the captured step never share an autograd graph or a parameter
        m_e, o_e = build(kw)
        tr = Trainer(m_e, torch.nn.BCELoss(), o_e)
        m_g, o_g = build(kw)
        gs = GraphedTrainStep(m_g, torch.nn.BCELoss(), o_g, warmup=1)
        k = {"i": 0}

        def eager(tr=tr, k=k):
            ins, y = pool[k["i"] % 4]
            k["i"] += 1
            tr.train_loop(*ins, train_rating=y)

        def graphed(gs=gs, k=k):
            ins, y = pool[k["i"] % 4]
            k["i"] += 1
            gs(*ins, rating=y)
        steps[f"{name} eager"] = eager
        steps[f"{name} graph-replayed"] = graphed
    t = run(steps, args.iters, args.rounds)
    emit(*report("2. DIEN train step (fused rows, SGD), per step", {f"{n} eager": t[f"{n} eager"] for n in variants}, "ms", 1.0,
                 "gru eager"))
    emit(*report("", {f"{n} graph-replayed": t[f"{n} graph-replayed"] for n in variants}, "ms", 1.0, "gru graph-replayed")[1:])
    ops.check_status()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(out) + "\n")


if __name__ == "__main__":
    main()
