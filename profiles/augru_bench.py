"""DIEN's AUGRU against the GRU at the C4 shape: B = 8192, L = 100, D = H = 64, one GPU.

1. Kernels: rs_augru_fwd / rs_augru_bwd against rs_gru_fwd / rs_gru_bwd, per call (training forward with the gate
   stash; backward from g_h_last).
2. The DIEN train step (1 M-row item table, fused sparse rows, SGD lr 0.01, Trainer.train_loop as bench.py --workload c4
   builds it) with evolution="gru" against evolution="augru", eager and CUDA-graph replayed (GraphedTrainStep).
3. The AUGRU recurrence forward + backward (input projection, L steps, BPTT, d att) as this package runs it
   (attention.augru_last_hidden) against the same recurrence written as a torch loop in fp32 with autograd on the GPU,
   the route a user of stock torch would take.

Times: CUDA events around `--iters` back-to-back calls or steps, repeated `--rounds` times with the variants alternating
inside every round; the median over rounds is printed (and the spread, min..max).  Every variant is warmed up first.
The step's working set (256 MB table, 8192 x 100 x 64 history rows) exceeds the 126 MB L2.

    python profiles/augru_bench.py [--iters 20] [--rounds 7] [--out FILE]
"""
import argparse
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from deeplearningrecommendationsystem_b200 import attention, ops  # noqa: E402

B, L, D, ITEMS, LR = 8192, 100, 64, 1_000_000, 0.01


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[torch.cuda.current_device()] if out else torch.cuda.get_device_name()
    except (OSError, subprocess.SubprocessError):
        return torch.cuda.get_device_name() + " (power limit not readable)"


def zipf_ids(c, shape, g, a=1.05):
    """bench.py's zipf ids: inverse CDF of a continuous power law with exponent a, truncated to [1, c]"""
    u = torch.rand(shape, generator=g, device="cuda", dtype=torch.float64)
    return ((((c ** (1 - a) - 1) * u + 1) ** (1 / (1 - a))).floor().long() - 1).clamp_(0, c - 1)


def timed(fn, iters):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / iters          # ms per call


def run(variants, iters, rounds, warmup=3):
    for fn in variants.values():
        for _ in range(warmup):
            fn()
    torch.cuda.synchronize()
    times = {k: [] for k in variants}
    for _ in range(rounds):
        for k, fn in variants.items():
            times[k].append(timed(fn, iters))
    return {k: sorted(v) for k, v in times.items()}


def report(title, times, unit="ms", scale=1.0, base=None):
    lines = [title]
    for k, v in times.items():
        med = v[len(v) // 2] * scale
        rel = f"   x{med / (times[base][len(times[base]) // 2] * scale):.3f} of {base}" if base and k != base else ""
        lines.append(f"  {k:40s} {med:9.3f} {unit}  (min {v[0] * scale:.3f}, max {v[-1] * scale:.3f}){rel}")
    return lines


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
    emit(f"card: {card()}", f"shape: B = {B}, L = {L}, D = H = {D}; {args.rounds} rounds x {args.iters} calls, medians", "")
    g = torch.Generator(device="cuda").manual_seed(0)
    H = D

    # 1. kernels
    gi = torch.randn(B, L, 3 * H, device="cuda", generator=g) * 0.5
    att = torch.softmax(torch.randn(B, L, device="cuda", generator=g), dim=1)
    w_hh = (torch.rand(3 * H, H, device="cuda", generator=g) * 2 - 1) / H ** 0.5
    b_hh = (torch.rand(3 * H, device="cuda", generator=g) * 2 - 1) / H ** 0.5
    gl = torch.randn(B, H, device="cuda", generator=g)
    h_g, gates_g = ops.gru_fwd(gi, w_hh, b_hh)
    h_a, gates_a = ops.augru_fwd(gi, att, w_hh, b_hh)
    t = run({"rs_gru_fwd": lambda: ops.gru_fwd(gi, w_hh, b_hh), "rs_augru_fwd": lambda: ops.augru_fwd(gi, att, w_hh, b_hh),
             "rs_gru_bwd": lambda: ops.gru_bwd(w_hh, h_g, gates_g, g_h_last=gl),
             "rs_augru_bwd": lambda: ops.augru_bwd(w_hh, att, h_a, gates_a, g_h_last=gl)}, args.iters * 5, args.rounds)
    emit(*report("1. recurrence kernels, per call", {k: t[k] for k in ("rs_gru_fwd", "rs_augru_fwd")}, "us", 1e3, "rs_gru_fwd"))
    emit(*report("", {k: t[k] for k in ("rs_gru_bwd", "rs_augru_bwd")}, "us", 1e3, "rs_gru_bwd")[1:])
    del gi, h_g, gates_g, h_a, gates_a
    emit("")

    # 2. the DIEN train step
    pool = []
    for _ in range(4):
        hist = zipf_ids(ITEMS, (B, L), g)
        tgt = torch.randint(0, ITEMS, (B,), generator=g, device="cuda")
        pool.append(((hist, tgt), (torch.rand(B, 1, generator=g, device="cuda") < 0.3).float()))
    steps = {}

    def build(evo):
        torch.manual_seed(0)
        m = M.DIEN(ITEMS, D, evolution=evo).cuda().fuse_embedding_updates()
        return m, FusedRowOptimizer(m, torch.optim.SGD([p for p in m.parameters() if p.requires_grad], lr=LR), lr=LR)
    for evo in ("gru", "augru"):
        # one model per leg: the eager and the captured step never share an autograd graph or a parameter
        m_e, o_e = build(evo)
        tr = Trainer(m_e, torch.nn.BCELoss(), o_e)
        m_g, o_g = build(evo)
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
        steps[f"DIEN {evo} eager"] = eager
        steps[f"DIEN {evo} graph-replayed"] = graphed
    t = run(steps, args.iters, args.rounds)
    emit(*report("2. DIEN train step (fused rows, SGD), per step", {k: t[k] for k in ("DIEN gru eager", "DIEN augru eager")},
                  "ms", 1.0, "DIEN gru eager"))
    emit(*report("", {k: t[k] for k in ("DIEN gru graph-replayed", "DIEN augru graph-replayed")}, "ms", 1.0,
                  "DIEN gru graph-replayed")[1:])
    ops.check_status()
    del steps, pool
    torch.cuda.empty_cache()
    emit("")

    # 3. the recurrence as a library call against a torch loop
    gru = torch.nn.GRU(D, H, batch_first=True).cuda()
    x = (torch.randn(B, L, D, device="cuda", generator=g) * 0.5).requires_grad_(True)
    a = att.clone().requires_grad_(True)

    def torch_loop():
        gi = torch.nn.functional.linear(x, gru.weight_ih_l0, gru.bias_ih_l0)
        h = x.new_zeros(B, H)
        for s in range(L):
            gh = torch.nn.functional.linear(h, gru.weight_hh_l0, gru.bias_hh_l0)
            ir, iz, inn = gi[:, s].chunk(3, dim=1)
            hr, hz, hn = gh.chunk(3, dim=1)
            r, z = torch.sigmoid(ir + hr), torch.sigmoid(iz + hz)
            n = torch.tanh(inn + r * hn)
            u = a[:, s:s + 1] * (1.0 - z)
            h = (1.0 - u) * h + u * n
        (h * gl).sum().backward()

    def library():
        (attention.augru_last_hidden(x, a, gru) * gl).sum().backward()
    with torch.no_grad():
        ref_h = attention.augru_last_hidden(x, a, gru)
    t = run({"augru_last_hidden (rs_augru_*)": library, "torch loop, fp32 autograd": torch_loop}, max(1, args.iters // 4), args.rounds)
    emit(*report("3. AUGRU recurrence forward + backward (projection GEMM, L steps, BPTT, d att), per call", t, "ms", 1.0,
                  "augru_last_hidden (rs_augru_*)"))
    # the two routes compute the same function (fp32 rounding apart)
    h_loop = x.new_zeros(B, H)
    with torch.no_grad():
        gi2 = torch.nn.functional.linear(x, gru.weight_ih_l0, gru.bias_ih_l0)
        for s in range(L):
            gh = torch.nn.functional.linear(h_loop, gru.weight_hh_l0, gru.bias_hh_l0)
            ir, iz, inn = gi2[:, s].chunk(3, dim=1)
            hr, hz, hn = gh.chunk(3, dim=1)
            r, z = torch.sigmoid(ir + hr), torch.sigmoid(iz + hz)
            n = torch.tanh(inn + r * hn)
            u = a[:, s:s + 1] * (1.0 - z)
            h_loop = (1.0 - u) * h_loop + u * n
    emit(f"  max |h_L(library) - h_L(torch loop)| = {float((ref_h - h_loop).abs().max()):.2e}")
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(out) + "\n")


if __name__ == "__main__":
    main()
