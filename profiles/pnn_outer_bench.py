"""The PNN paper's outer-product layer (FieldPNN(product="outer")) at the C3 shape: B = 32768, 39 fields, D = 32, H0 = 256.

1. Kernels: rs_pnn_outer_fwd (weight repack + qf_kernel) and rs_pnn_outer_bwd (repack + qf_kernel for dS + wgrad_kernel +
   slab reduce) per call, CUDA events.  The split of the backward into its kernels comes from a separate torch.profiler
   run (kernel durations summed per name over the profiled calls).  Each contraction is 2 B H0 D^2 = 17.2 GFLOP
   (logical, one MAC = 2 FLOP; 3xTF32 issues three times that on the tensor cores); the share printed is of the
   1,125 TFLOP/s dense TF32 figure of NVIDIA's B200 data sheet, a data-sheet rate, not a measured one.
2. The same layer composed from torch ops on the same GPU: s = E.sum(1), materialised p = vec(s s^T) (B x D^2), an fp32
   nn.Linear (torch's default: no TF32), autograd for the backward; output agreement on the same seeded inputs.
3. The C3 train step (Trainer.train_loop, FusedRowOptimizer over torch SGD as bench.py builds it) with product="inner"
   and product="outer", eager and graph-replayed (GraphedTrainStep), the four variants alternating inside each round.

Times: medians over `--rounds` rounds of `--iters` back-to-back calls (min..max in brackets); every variant warmed up.
The train steps' working set (4.3 GB table per model) exceeds the 126 MB L2; the layer's inputs (E: 164 MB) do too.

    python profiles/pnn_outer_bench.py [--iters 20] [--rounds 7] [--out FILE]
"""
import argparse
import os
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from augru_bench import card, report, run  # noqa: E402
from deeplearningrecommendationsystem_b200 import ops  # noqa: E402

CRITEO = [1460, 583, 10131227, 2202608, 305, 24, 12517, 633, 3, 93145, 5683, 8351593, 3194, 27, 14992, 5461306, 10, 5652,
          2173, 4, 7046547, 18, 15, 286181, 105, 142572]
CARDS = CRITEO + [64] * 13
B, D, HIDDEN, LR = 32768, 32, [256, 128, 64, 32], 0.05
TF32_DATASHEET = 1125e12


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--out", default=None, help="also write the report to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a GPU")
    from deeplearningrecommendationsystem_b200.graph import GraphedTrainStep
    from deeplearningrecommendationsystem_b200.nfield import FieldPNN
    from deeplearningrecommendationsystem_b200.optim import FusedRowOptimizer
    from deeplearningrecommendationsystem_b200.trainer import Trainer
    out = []

    def emit(*lines):
        for line in lines:
            print(line, flush=True)
            out.append(line)
    F, H0 = len(CARDS), HIDDEN[0]
    flop = 2.0 * B * H0 * D * D
    emit(f"card: {card()}", f"shape: B = {B}, F = {F}, D = {D}, H0 = {H0}; {args.rounds} rounds x {args.iters} calls, medians",
         f"one contraction = 2 B H0 D^2 = {flop / 1e9:.1f} GFLOP (logical); shares are of the 1,125 TFLOP/s TF32 data-sheet rate", "")
    g = torch.Generator(device="cuda").manual_seed(0)
    E = torch.randn(B, F, D, device="cuda", generator=g) * (0.5 / F ** 0.5)
    W = torch.randn(H0, D * D, device="cuda", generator=g) / D
    bias = torch.randn(H0, device="cuda", generator=g) * 0.1
    gl = torch.randn(B, H0, device="cuda", generator=g) * 1e-3
    lp, S = ops.pnn_outer_fwd(E, W, bias)

    # 1 + 2. kernels, and the torch composition
    Et = E.clone().requires_grad_(True)
    lin = torch.nn.Linear(D * D, H0).cuda()
    with torch.no_grad():
        lin.weight.copy_(W)
        lin.bias.copy_(bias)

    def torch_fwd():
        s = Et.sum(1)
        return lin((s.unsqueeze(2) * s.unsqueeze(1)).reshape(B, D * D))

    def torch_fwd_bwd():
        Et.grad = lin.weight.grad = lin.bias.grad = None
        torch_fwd().backward(gl)
    t = run({"rs_pnn_outer_fwd": lambda: ops.pnn_outer_fwd(E, W, bias), "rs_pnn_outer_bwd": lambda: ops.pnn_outer_bwd(S, gl, W),
             "torch forward": lambda: torch_fwd(), "torch forward + backward": torch_fwd_bwd}, args.iters, args.rounds)
    emit(*report("1. the layer's kernels, per call", {k: t[k] for k in ("rs_pnn_outer_fwd", "rs_pnn_outer_bwd")}, "ms"))
    med = {k: v[len(v) // 2] for k, v in t.items()}
    emit(f"  forward: {flop / (med['rs_pnn_outer_fwd'] * 1e-3) / 1e12:.1f} TFLOP/s logical "
         f"({100 * flop / (med['rs_pnn_outer_fwd'] * 1e-3) / TF32_DATASHEET:.1f}% of the TF32 data-sheet rate)")
    emit(f"  backward (dS and dW, two contractions): {2 * flop / (med['rs_pnn_outer_bwd'] * 1e-3) / 1e12:.1f} TFLOP/s logical "
         f"({100 * 2 * flop / (med['rs_pnn_outer_bwd'] * 1e-3) / TF32_DATASHEET:.1f}% of the TF32 data-sheet rate)")
    # per-kernel split from a separate profiled run
    from torch.profiler import ProfilerActivity, profile
    n_prof = 5
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(n_prof):
            ops.pnn_outer_fwd(E, W, bias)
            ops.pnn_outer_bwd(S, gl, W)
        torch.cuda.synchronize()
    per = {}
    for ev in prof.events():
        if ev.device_type == torch.autograd.DeviceType.CUDA:
            per[ev.name] = per.get(ev.name, 0.0) + ev.device_time / n_prof
    emit("  kernels (torch.profiler, mean over the profiled calls):")
    for name, us in sorted(per.items(), key=lambda kv: -kv[1]):
        short = name.replace("(anonymous namespace)::", "").replace("void ", "").split("(")[0]
        rate = ""
        if short.startswith("qf_kernel") or short.startswith("wgrad_kernel"):
            r = flop / (us * 1e-6)
            what = "forward" if "false" in short else ("backward data" if "true" in short else "weight gradient")
            rate = f"   {what}: {r / 1e12:.1f} TFLOP/s logical, {100 * r / TF32_DATASHEET:.1f}% of the data-sheet rate"
        emit(f"    {short:34s} {us:9.1f} us{rate}")
    emit("")
    emit(*report("2. the layer composed from torch ops (materialised p, fp32 nn.Linear, autograd), per call",
                 {k: t[k] for k in ("torch forward", "torch forward + backward")}, "ms"))
    kern = med["rs_pnn_outer_fwd"] + med["rs_pnn_outer_bwd"]
    emit(f"  forward: kernels x{med['torch forward'] / med['rs_pnn_outer_fwd']:.2f} faster; forward + backward: "
         f"{kern:.3f} ms against {med['torch forward + backward']:.3f} ms (x{med['torch forward + backward'] / kern:.2f})")
    torch_fwd_bwd()
    dS, dW, db = ops.pnn_outer_bwd(S, gl, W)
    with torch.no_grad():
        lp_t = torch_fwd()
    rel = lambda a, b: float((a - b).abs().max() / b.abs().max())   # noqa: E731
    emit(f"  agreement, max |kernel - torch| / max |torch|: lp {rel(lp, lp_t):.2e}, dE {rel(dS, Et.grad[:, 0]):.2e}, "
         f"dW {rel(dW, lin.weight.grad):.2e}, db {rel(db, lin.bias.grad):.2e}")
    del Et, lin, E, S, lp, lp_t, dS, dW, db
    torch.cuda.empty_cache()
    emit("")

    # 3. the C3 train step
    pool = []
    for _ in range(4):
        ids = torch.stack([torch.randint(0, c, (B,), generator=g, device="cuda") for c in CARDS], dim=1).contiguous()
        pool.append((ids, (torch.rand(B, 1, generator=g, device="cuda") < 0.3).float()))

    def build(product):
        torch.manual_seed(0)
        m = FieldPNN(CARDS, D, HIDDEN, seed=1, device="cuda", product=product)
        return m, FusedRowOptimizer(m, torch.optim.SGD([p for p in m.parameters() if p.requires_grad], lr=LR), lr=LR, kind="sgd")
    steps = {}
    for product in ("inner", "outer"):
        m_e, o_e = build(product)
        tr = Trainer(m_e, torch.nn.BCELoss(), o_e)
        m_g, o_g = build(product)
        gs = GraphedTrainStep(m_g, torch.nn.BCELoss(), o_g, warmup=1)
        k = {"i": 0}

        def eager(tr=tr, k=k):
            ids, y = pool[k["i"] % 4]
            k["i"] += 1
            tr.train_loop(ids, train_rating=y)

        def graphed(gs=gs, k=k):
            ids, y = pool[k["i"] % 4]
            k["i"] += 1
            gs(ids, rating=y)
        steps[f"C3 {product} eager"] = eager
        steps[f"C3 {product} graph-replayed"] = graphed
    t = run(steps, args.iters, args.rounds)
    emit(*report("3. C3 FieldPNN train step (fused rows, SGD), per step", {k: t[k] for k in ("C3 inner eager", "C3 outer eager")}, "ms",
                 1.0, "C3 inner eager"))
    emit(*report("", {k: t[k] for k in ("C3 inner graph-replayed", "C3 outer graph-replayed")}, "ms", 1.0, "C3 inner graph-replayed")[1:])
    ops.check_status()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(out) + "\n")


if __name__ == "__main__":
    main()
