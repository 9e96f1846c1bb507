"""rs_replica_sgd vs rs_replica_update (SGD with weight decay, Adam) on the C2 replicated sub-table, one GPU.

The shape is what the hybrid placement replicates at C2: the 18 Criteo-Kaggle fields under 65 536 rows, 47 398 rows, at
W = 416 (FFM rows, 78.9 MB) and W = 16 (FM rows, 3.0 MB).  Touched flags come from a uniform batch of 65 536 samples per
rank over those fields, as the C2 benchmark draws its ids.

world = 1: one rank updates the whole table.  world = 8: all eight ranks' replicas, gradients and flags live on this one
GPU and only rank 0's launch (one eighth of the table) is timed -- a LOCAL-MEMORY PROXY for the NVLink case: its peer loads
and stores go to HBM, not over NVLink, so it bounds neither the real 8-GPU time nor its link traffic.

Times: CUDA events around `--launches` back-to-back launches, repeated `--rounds` times with the variants alternating;
the median per launch is printed.  Bytes are computed from shapes (slice floats x bytes per float; flag bytes added for
the lazy kernels).  The W = 416 working set (w + g, and m + v for Adam) is close to or above the 126 MB L2; W = 16 sits
in L2.

    python profiles/replica_update_bench.py [--launches 200] [--rounds 5]
"""
import argparse
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from deeplearningrecommendationsystem_b200 import ops  # noqa: E402

C2 = [1460, 583, 10131227, 2202608, 305, 24, 12517, 633, 3, 93145, 5683, 8351593, 3194, 27, 14992, 5461306, 10, 5652, 2173,
      4, 7046547, 18, 15, 286181, 105, 142572]
SMALL = [c for c in C2 if c < 65536]
B = 65536


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[torch.cuda.current_device()] if out else torch.cuda.get_device_name()
    except (OSError, subprocess.SubprocessError):
        return torch.cuda.get_device_name() + " (power limit not readable)"


def flags_for(rank):
    g = torch.Generator().manual_seed(100 + rank)
    t = torch.zeros(sum(SMALL), dtype=torch.uint8)
    off = 0
    for c in SMALL:
        t[off + torch.randint(0, c, (B,), generator=g)] = 1
        off += c
    return t.cuda()


def timed(fn, launches):
    fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(launches):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / launches * 1e3          # us per launch


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a GPU")
    rows = sum(SMALL)
    print(f"card: {card()}")
    print(f"C2 replicated sub-table: {len(SMALL)} fields, {rows} rows")
    for world in (1, 8):
        flags = [flags_for(r) for r in range(world)]
        any_hit = torch.stack(flags).any(0)
        for W in (416, 16):
            numel = rows * W
            g = torch.Generator(device="cuda").manual_seed(W)
            w = [torch.randn(numel, device="cuda", generator=g) * 0.01 for _ in range(world)]
            gr = [torch.randn(numel, device="cuda", generator=g) * 1e-3 for _ in range(world)]
            wp, gp, fp = [t.data_ptr() for t in w], [t.data_ptr() for t in gr], [t.data_ptr() for t in flags]
            lo, hi = ops.replica_slice(numel, world, 0)
            m, v = torch.zeros(hi - lo, device="cuda"), torch.zeros(hi - lo, device="cuda")
            n = hi - lo
            hit_frac = float(any_hit.repeat_interleave(W)[lo:hi].float().mean())
            base = (2 * world + 1) * 4 * n                         # world gradient reads, own w read, world w stores
            flag_bytes = world * (hi - lo) // W                    # one flag per rank per row of the slice
            variants = {
                "rs_replica_sgd": (lambda: ops.replica_sgd(wp, gp, numel, world, 0, 1e-6), base),
                "rs_replica_update sgd+wd": (lambda: ops.replica_update(wp, gp, fp, numel, W, world, 0, "sgd", 1e-6, 1e-5),
                                             base * hit_frac + flag_bytes),
                "rs_replica_update adam+wd": (lambda: ops.replica_update(wp, gp, fp, numel, W, world, 0, "adam", 1e-6, 1e-5, m=m, v=v, step=1),
                                              (base + 16 * n) * hit_frac + flag_bytes),
            }
            times = {k: [] for k in variants}
            for _ in range(args.rounds):
                for k, (fn, _) in variants.items():
                    times[k].append(timed(fn, args.launches))
            torch.cuda.synchronize()
            label = "one GPU" if world == 1 else "8 ranks on one GPU, rank 0's slice (local-memory proxy for NVLink)"
            print(f"\nworld {world} ({label}), W = {W}: table {numel * 4 / 1e6:.1f} MB, slice {n * 4 / 1e6:.2f} MB, "
                  f"rows touched by some rank {hit_frac:.3f}")
            for k, (_, nbytes) in variants.items():
                t = sorted(times[k])[len(times[k]) // 2]
                print(f"  {k:28s} {t:8.1f} us   {nbytes / 1e6:8.2f} MB   {nbytes / t / 1e6:6.2f} TB/s")
            ops.check_status()


if __name__ == "__main__":
    main()
