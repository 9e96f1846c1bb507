#!/usr/bin/env python
"""Benchmark of the embedding -> interaction -> sparse-update hot path on B200 (contract: the task brief, section 4).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c2|c1|c3|c4|c5|rank] [--impl reference] [--dist uniform|zipf]
                    [--dump-outputs DIR]

Default workload = BASELINE.json configs[1] ("C2", the config the metric is quoted on): FM second-order + FFM on synthetic
Criteo-shaped data -- 26 sparse fields, D = 16, batch 65536 per GPU, the public Criteo-Kaggle cardinalities (33.76 M rows;
FFM table 56.2 GB, FM table 2.2 GB), uniform ids, Bernoulli(0.3) labels, plain SGD.  One "step" = one FFM train step + one
FM train step over the same batch through the public API (model -> BCELoss -> backward -> FusedRowOptimizer.step(), i.e.
Trainer.train_loop).  N > 1: one process per GPU, tables row-sharded, exchange through dist.DeviceRowExchange.

Every workload prints ONE JSON line per model with
  value         whole-job samples/s, inputs resident in HBM (eager Trainer.train_loop, kernels bracketed by CUDA events)
  e2e           same metric from pinned HOST buffers: H2D of ids/labels and D2H of the loss inside the timed region
  roofline      dominant kernel: algorithmic bytes (or logical FLOPs) of one launch / its CUDA-event duration vs MEASURED_PEAKS.json
  cpu_baseline  N = 1 only: the reference's CPU implementation of the path timed on this box's host cores (bounded sample)
  clocks, gpu_launches, and -- default workload only -- "zipf", "light", "c5" and (N > 1) "sharded_equals_single" sub-records.
`--impl reference` times the CPU arm alone: the unmodified reference classes from oracle/_ref (byte-compiled by
oracle/build_ref.py) for c1 / c4 / c5, the validated N-field oracle port for c2 / c3 (the reference modules are hard-wired
to six MovieLens features).
"""
import argparse
import json
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CRITEO = [1460, 583, 10131227, 2202608, 305, 24, 12517, 633, 3, 93145, 5683, 8351593, 3194, 27, 14992, 5461306, 10, 5652,
          2173, 4, 7046547, 18, 15, 286181, 105, 142572]
F, D, BATCH = 26, 16, 65536
LR = 0.05
METRIC = "train samples/sec (fwd+bwd+update)"
WORKLOADS = {
    "c2": "C2: FM second-order + FFM train step, 26 Criteo-shaped sparse fields, D=16, batch 65536, SGD",
    "c1": "C1: DeepFM on MovieLens-100k shapes (scripts/deepfm.py: B=87909 full batch, D=128, hidden [512,256,128,1], Adam 1e-3 wd 1e-5)",
    "c3": "C3: PNN inner product / AFM attention pooling, 39 fields, D=32, batch 32768",
    "c4": "C4: DIN / DIEN target attention, behaviour seq len 100, D=64, batch 8192",
    "c5": "C5: MF / NeuralCF with 100 M-row user and item tables, batch 65536 per GPU",
}
NOMINAL_HBM_GBS = 8000.0          # the ~8 TB/s the north star quotes


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    out = {"hbm_gbs": 6650.0, "bf16_tflops_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        out.update(hbm_gbs=d.get("hbm_gbs", out["hbm_gbs"]), bf16_tflops_sustained=d.get("bf16_tflops_sustained", d.get("bf16_tflops", 1400.0)),
                   source="measured (MEASURED_PEAKS.json)")
    return out


def zipf_ids(c, shape, g, device, a=1.05):
    """inverse CDF of a continuous power law with exponent a, truncated to [1, c]"""
    u = torch.rand(shape, generator=g, device=device, dtype=torch.float64)
    x = ((c ** (1 - a) - 1) * u + 1) ** (1 / (1 - a))
    return (x.floor().long() - 1).clamp_(0, c - 1)


def make_ids(cards, B, seed, dist, device):
    g = torch.Generator(device=device).manual_seed(seed)
    cols = [zipf_ids(c, (B,), g, device) if dist == "zipf" else torch.randint(0, c, (B,), generator=g, device=device) for c in cards]
    ids = torch.stack(cols, dim=1).contiguous()
    y = (torch.rand(B, 1, generator=g, device=device) < 0.3).float()
    return ids, y


class ClockSampler:
    """Samples SM clock and throttle reasons through NVML every few ms on a background thread while the timed
    region runs (the same counters `nvidia-smi --query-gpu=clocks.sm,clocks_event_reasons.*` prints)."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index, period_s=float(os.environ.get("RS_BENCH_CLOCK_PERIOD", "0.004"))):
        import threading
        self.sm, self.mask, self.max_mhz, self.ok = [], 0, None, False
        self._stop = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(visible.split(",")[index]) if visible and visible.split(",")[index].isdigit() else index
            self.nv, self.h = pynvml, pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception:
            return
        self.period = period_s
        self.t = threading.Thread(target=self._run, daemon=True)
        self.t.start()

    def _run(self):
        while not self._stop.is_set():
            try:
                self.sm.append(float(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)))
                self.mask |= int(self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
            except Exception:
                pass
            self._stop.wait(self.period)

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        if not self.ok:
            return out
        self._stop.set()
        self.t.join(timeout=2)
        if self.sm:
            v = sorted(self.sm)
            out.update(sm_mhz=v[len(v) // 2], samples=len(v), reasons=sorted(n for bit, n in self.REASONS.items() if self.mask & bit))
        return out


def progress(msg):
    """stage markers on stderr (rank 0): a hung multi-GPU run can then be located from its log"""
    if int(os.environ.get("RANK", "0")) == 0:
        print(f"[bench {time.strftime('%H:%M:%S')}] {msg}", file=sys.stderr, flush=True)


def env():
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return world, rank, local


# ====================================================================================================== CPU arm
def _ref_modules():
    try:
        from oracle.build_ref import import_ref
        return import_ref()
    except Exception:
        return None


def cpu_step_factory(workload, model, threads, light=True):
    """-> (step() -> loss float, samples per step, kind, sample description).  The reference's CPU implementation of one
    train step of `workload`: the UNMODIFIED reference classes (oracle/_ref, kind "reference") where they are
    size-generic (c1 DeepFM; c4 DIN / DIEN; c5 MF / NeuralCF at 1 M rows -- 100 M rows cannot be instantiated with a dense
    gradient), else the validated N-field oracle port (c2, c3: the reference modules are hard-wired to six features)."""
    torch.set_num_threads(threads)
    g = torch.Generator().manual_seed(0)
    ref = _ref_modules()
    bce = torch.nn.BCELoss()
    if workload == "c2":
        from oracle import nfield as onf
        cap = 1 << 17
        cards = [min(c, cap) for c in CRITEO]
        B = BATCH
        offsets = torch.tensor([sum(cards[:i]) for i in range(F)])
        total = sum(cards)
        fm_t, ffm_t = torch.randn(total, D, generator=g) * 0.01, torch.randn(total, F * D, generator=g) * 0.01
        fm_b, ffm_b = torch.zeros(1), torch.zeros(1)
        ids = torch.stack([torch.randint(0, c, (B,), generator=g) for c in cards], dim=1)
        y = (torch.rand(B, generator=g) < 0.3).float()

        def step():
            onf.train_step("fm", fm_t, fm_b, ids, offsets, y, LR)
            _, loss = onf.train_step("ffm", ffm_t, ffm_b, ids, offsets, y, LR, fast=True)
            return float(loss)
        return step, B, "port", (f"full batch B={B}, 26 fields, D=16, cardinalities capped at 2^17 rows/field ({total} rows; the GPU line's "
                                 "'light' sub-record runs this same config), nn.Embedding-style dense gradient + dense SGD, oracle/nfield.py")
    if workload == "c3":
        from oracle import nfield as onf
        cards = [min(c, 1 << 17) for c in CRITEO] + [64] * 13
        B = 4096
        ids = torch.stack([torch.randint(0, c, (B,), generator=g) for c in cards], dim=1)
        y = (torch.rand(B, 1, generator=g) < 0.3).float()
        m = onf.PortPNN(cards, 32, [256, 128, 64, 32]) if model == "PNN-inner" else onf.PortAFM(cards, 32, 64)
        opt = torch.optim.SGD(m.parameters(), lr=LR)

        def step():
            opt.zero_grad()
            loss = bce(m(ids), y)
            loss.backward()
            opt.step()
            return float(loss.detach())
        return step, B, "port", (f"B={B} of 32768, 39 fields, D=32, cardinalities capped at 2^17, dense-gradient SGD, oracle/nfield.Port{model[:3]}")
    # ---- the real reference classes
    kind = "reference" if ref is not None else "port"
    if workload == "c1":
        B = 87909
        x = feature_matrix_fast(g, B, 943, 1682)
        y = (torch.rand(B, 1, generator=g) < 0.3).float()
        if ref is not None:
            m = ref["model.deepfm"].DeepFM(943, 1682, [512, 256, 128, 1], 128)
            opt = torch.optim.Adam(m.parameters(), lr=1e-3, weight_decay=1e-5)
            tr = ref["trainer.trainer"].Trainer(m, bce, opt)

            def step():
                tr.train_loop(x, train_rating=y)
                return float(tr.train_loss.detach())
        else:                                      # oracle port of the same model (oracle/ml100k.py) + torch Adam
            from oracle import ml100k
            from deeplearningrecommendationsystem_b200.model import DeepFM
            sd = {k: v.detach().clone().requires_grad_(True) for k, v in DeepFM(943, 1682, [512, 256, 128, 1], 128).state_dict().items()}
            opt = torch.optim.Adam(list(sd.values()), lr=1e-3, weight_decay=1e-5)

            def step():
                opt.zero_grad()
                loss = bce(ml100k.forward("deepfm", sd, x), y)
                loss.backward()
                opt.step()
                return float(loss.detach())
        return step, B, kind, "full batch B=87909 x 45 synthetic ML-100k-shaped features; reference model/deepfm.py + trainer/trainer.py + optim.Adam(1e-3, wd=1e-5)"
    if ref is None:
        raise RuntimeError("oracle/_ref missing: run `python oracle/build_ref.py` where the reference tree is mounted")
    if workload == "c4":
        B, L, items = 8192, 100, 1_000_000
        hist = zipf_ids(items, (B, L), g, "cpu")
        tgt = torch.randint(0, items, (B,), generator=g)
        y = (torch.rand(B, 1, generator=g) < 0.3).float()
        m = (ref["model.din"].DIN if model == "DIN" else ref["model.dien"].DIEN)(items, 64)
        opt = torch.optim.SGD(m.parameters(), lr=0.01)
        tr = ref["trainer.trainer"].Trainer(m, bce, opt)

        def step():
            tr.train_loop(hist, tgt, train_rating=y)
            return float(tr.train_loss.detach())
        return step, B, kind, f"full batch B={B}, L=100, D=64, 1 M-row item table; reference model/{model.lower()}.py + Trainer + dense optim.SGD"
    if workload == "c5":
        rows, B = 1_000_000, 65536
        u, i = torch.randint(0, rows, (B,), generator=g), torch.randint(0, rows, (B,), generator=g)
        if model == "MF":
            m, y = ref["model.mf"].MatrixFactorization(rows, rows, 64), (torch.rand(B, generator=g) < 0.3).float()
        else:
            m, y = ref["model.neuralcf"].NeuralCF(rows, rows, 64, [128, 64, 32, 16]), (torch.rand(B, 1, generator=g) < 0.3).float()
        opt = torch.optim.SGD(m.parameters(), lr=LR)
        tr = ref["trainer.trainer"].Trainer(m, bce, opt)

        def step():
            tr.train_loop(u, i, train_rating=y)
            return float(tr.train_loss.detach())
        return step, B, kind, (f"full batch B={B}, tables of 1 M rows instead of 100 M (a dense gradient + dense SGD sweep over 100 M x 64 "
                               f"rows does not fit the host), D=64; reference model/{'mf' if model == 'MF' else 'neuralcf'}.py + Trainer + optim.SGD")
    raise ValueError(workload)


def feature_matrix_fast(g, B, nu, ni):
    """(B,45) float32 in the data/reader.py:98-101 column order (vectorised: tests/helpers.feature_matrix loops over B)"""
    x = torch.zeros(B, 45)
    x[:, 0] = torch.randint(0, nu, (B,), generator=g).float()
    x[:, 1] = torch.randint(0, ni, (B,), generator=g).float()
    x[:, 2] = torch.rand(B, generator=g)
    r = torch.arange(B)
    x[r, 3 + torch.randint(0, 2, (B,), generator=g)] = 1.0
    x[r, 5 + torch.randint(0, 21, (B,), generator=g)] = 1.0
    n_genre = torch.randint(0, 7, (B, 1), generator=g)
    order = torch.rand(B, 19, generator=g).argsort(dim=1)
    x[:, 26:] = (order < n_genre).float()            # n_genre distinct random genres per row
    return x


def time_cpu(workload, model, steps, warmup):
    threads = os.cpu_count() or 1
    step, B, kind, sample = cpu_step_factory(workload, model, threads)
    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        loss = step()
    dt = (time.perf_counter() - t0) / steps
    return {"value": B / dt, "unit": "samples/s", "cores": threads, "kind": kind, "sample": sample, "ms_per_step": dt * 1e3, "last_loss": loss}


MODELS_OF = {"c1": ["DeepFM"], "c2": ["FM+FFM"], "c3": ["PNN-inner", "AFM"], "c4": ["DIN", "DIEN"], "c5": ["MF", "NeuralCF"]}


def run_reference(args):
    world, rank, _ = env()
    if rank != 0:
        return
    for model in MODELS_OF[args.workload]:
        # bounded: one warm-up + at most three timed steps of the sample (each step is seconds of host work)
        cb = time_cpu(args.workload, model, max(1, min(args.steps, 3)), 1)
        line = {
            "impl": "reference", "metric": METRIC, "value": cb["value"], "unit": "samples/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": cb["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOADS[args.workload] + ("" if len(MODELS_OF[args.workload]) == 1 else f" [{model}]"), "sample": cb["sample"],
                       "impl": "reference CPU path (torch CPU fp32, all host threads)", "timed_steps": max(1, min(args.steps, 3))},
            "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": cb["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
        }
        print(json.dumps(line), flush=True)


# ====================================================================================================== GPU legs
def run_legs(step, pool, B, args, world, dev, local, graph_step=None, extra_warmup=0, e2e_steps=None, after_timed=None):
    """Device-resident leg (eager, per-kernel CUDA events, launch count) + end-to-end leg (inputs from pinned host memory on a
    copy stream, loss copied back every step; `graph_step` replays the same step as a CUDA graph when given).
    step(inputs tuple, y) -> loss tensor.  `after_timed()` runs once right after the timed steps, before any further step
    changes the models.  Returns a dict of raw measurements (times already max-reduced over ranks)."""
    import torch.distributed as dist
    from deeplearningrecommendationsystem_b200 import ops

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for k in range(args.warmup + extra_warmup):
        step(*pool[k % len(pool)])
    ops.check_status(dev)
    progress("  warm-up done")
    clocks = ClockSampler(local)
    sync()
    launches0 = ops.launches()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(args.steps):
        loss = step(*pool[k % len(pool)])
    e1.record()
    sync()
    ms_total = e0.elapsed_time(e1)
    gpu_launches = ops.launches() - launches0
    last_loss_eager = float(loss.detach())
    if after_timed is not None:
        after_timed()
    # per-kernel CUDA-event times come from a few EXTRA steps outside the timed region: bracketing every C-ABI call with two
    # events costs host time that the timed steps should not pay
    n_prof = min(args.steps, 5)
    ops.PROFILE = []
    for k in range(n_prof):
        loss = step(*pool[k % len(pool)])
    sync()
    prof, ops.PROFILE = ops.PROFILE, None
    del loss            # keeps the eager autograd graph (AccumulateGrad nodes bound to this stream) alive otherwise: breaks capture

    progress("  eager leg done")
    run = step
    api = "trainer.Trainer.train_loop (eager)"
    if graph_step is not None:
        run, api = graph_step, "graph.GraphedTrainStep (CUDA graph replay of the same step)"
        for k in range(3):                              # untimed: eager warm-up call(s), the capture, one replay
            run(*pool[k % len(pool)])
        progress("  graph captured")
    host_pool = [(tuple(t.cpu().pin_memory() for t in ins), y.cpu().pin_memory()) for ins, y in pool]
    copy_stream = torch.cuda.Stream(device=dev)
    main = torch.cuda.current_stream()
    slots = [(tuple(torch.empty_like(t) for t in pool[0][0]), torch.empty_like(pool[0][1])) for _ in range(2)]
    copied = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]
    h2d_events = []
    n_e2e = e2e_steps or args.steps

    def fetch(k):
        hins, hy = host_pool[k % len(host_pool)]
        b = k & 1
        with torch.cuda.stream(copy_stream):
            if k >= 2:
                copy_stream.wait_event(consumed[b])        # the step that read this slot has finished
            c0 = torch.cuda.Event(enable_timing=True)
            c0.record(copy_stream)
            for dst, src in zip(slots[b][0], hins):
                dst.copy_(src, non_blocking=True)
            slots[b][1].copy_(hy, non_blocking=True)
            c1 = torch.cuda.Event(enable_timing=True)
            c1.record(copy_stream)
            copied[b].record(copy_stream)
            h2d_events.append((c0, c1))

    loss_host = torch.zeros(n_e2e, dtype=torch.float32).pin_memory()
    sync()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    fetch(0)
    for k in range(n_e2e):
        b = k & 1
        if k + 1 < n_e2e:
            fetch(k + 1)
        main.wait_event(copied[b])
        loss_host[k:k + 1].copy_(run(*slots[b]).detach().reshape(1), non_blocking=True)
        consumed[b].record(main)
    t1.record()
    sync()
    ms_e2e = t0.elapsed_time(t1)
    clk = clocks.stop()
    ops.check_status(dev)
    h2d_ms = sorted(a.elapsed_time(b) for a, b in h2d_events)
    times = torch.tensor([ms_total / args.steps, ms_e2e / n_e2e], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    ms_step, ms_e2e_step = times.tolist()
    agg = {}
    for name, a, b in prof:
        agg.setdefault(name, []).append(a.elapsed_time(b))
    h2d_bytes = sum(t.numel() * t.element_size() for t in pool[0][0]) + pool[0][1].numel() * pool[0][1].element_size()
    return {"ms_step": ms_step, "ms_e2e": ms_e2e_step, "kern": {k: sum(v) / len(v) for k, v in agg.items()},
            "calls": {k: len(v) / n_prof for k, v in agg.items()}, "gpu_launches": gpu_launches, "clocks": clk,
            "last_loss": float(loss_host[-1]), "last_loss_eager": last_loss_eager, "e2e_api": api, "h2d_bytes": h2d_bytes,
            "h2d_copy_ms": {"median": h2d_ms[len(h2d_ms) // 2], "max": h2d_ms[-1]}, "e2e_steps": n_e2e}


def base_line(args, world, B, legs, workload, config):
    return {
        "metric": METRIC, "value": world * B / (legs["ms_step"] / 1e3), "unit": "samples/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": legs["ms_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": {"workload": workload, "batch_per_gpu": B, **config,
                                                         "step_api": "trainer.Trainer.train_loop (eager)",
                                                         "parallelism": f"dp{world}"},
        "e2e": {"value": world * B / (legs["ms_e2e"] / 1e3), "unit": "samples/s", "h2d_bytes_per_step": legs["h2d_bytes"],
                "d2h_bytes_per_step": 4, "ms_per_step": legs["ms_e2e"], "last_loss": legs["last_loss"], "step_api": legs["e2e_api"],
                "h2d_copy_ms": legs["h2d_copy_ms"], "steps": legs["e2e_steps"]},
        "gpu_launches": legs["gpu_launches"], "clocks": legs["clocks"],
        "kernels": {k: {"ms": v, "calls_per_step": legs["calls"][k]} for k, v in legs["kern"].items()},
    }


def hbm_roofline(kernel, what, bytes_per_launch, ms, traffic=None, note=None):
    pk = peaks()
    achieved = bytes_per_launch / (ms / 1e3) / 1e9
    out = {"bound": "hbm", "kernel": kernel, "achieved": achieved, "peak": pk["hbm_gbs"], "peak_source": pk["source"], "unit": "GB/s",
           "frac": achieved / pk["hbm_gbs"], "frac_of_nominal_8TBps": achieved / NOMINAL_HBM_GBS, "traffic": traffic,
           "algorithmic_bytes_per_launch": bytes_per_launch, "algorithmic_bytes": what, "ms_per_launch": ms}
    if note:
        out["note"] = note
    return out


def tensor_roofline(kernel, what, flops_per_launch, ms, passes=3):
    """3xTF32 kernels: logical fp32 FLOPs against the tf32 pipe (= measured dense bf16 / 2) divided by the `passes` MMAs
    each logical MAC costs."""
    pk = peaks()
    peak = pk["bf16_tflops_sustained"] / 2.0 / passes
    achieved = flops_per_launch / (ms / 1e3) / 1e12
    return {"bound": "tensor", "kernel": kernel, "achieved": achieved, "peak": peak, "peak_source": pk["source"] + f": bf16 sustained / 2 (tf32) / {passes} (3xTF32 split)",
            "unit": "TFLOP/s", "frac": achieved / peak, "traffic": None, "logical_flops_per_launch": flops_per_launch, "flops": what, "ms_per_launch": ms}


def ncu_traffic(key):
    """DRAM bytes per launch of `key` from the committed ncu capture (profiles/ncu_traffic.json), or None."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    try:
        with open(p) as f:
            return json.load(f).get(key)
    except Exception:
        return None


# ====================================================================================================== C2 (headline)
def build_c2(cards, dev, world, exchange=None, fabric=None):
    from deeplearningrecommendationsystem_b200.nfield import FieldFFM, FieldFM
    from deeplearningrecommendationsystem_b200.optim import FusedRowOptimizer
    from deeplearningrecommendationsystem_b200.trainer import Trainer
    sharded = world > 1 or exchange is not None or os.environ.get("RS_BENCH_FORCE_SHARDED") == "1"   # world 1: same kernels, local "peers"
    if sharded and exchange is None:
        from deeplearningrecommendationsystem_b200 import dist as rsdist
        from deeplearningrecommendationsystem_b200.nfield import REPLICATE_ROWS, direct_ranges
        # default placement: tables under REPLICATE_ROWS rows are replicated, the others row-sharded (nfield._FieldModel);
        # RS_REPLICATE_ROWS=0 row-shards every table (then the largest fields are read directly by the FFM forward)
        rep = int(os.environ.get("RS_REPLICATE_ROWS", REPLICATE_ROWS))
        hybrid = any(c < rep for c in cards) and any(c >= rep for c in cards)
        direct = direct_ranges(cards) if (os.environ.get("RS_DIRECT", "1") == "1" and not hybrid) else ()
        exchange = rsdist.DeviceRowExchange(fabric, direct=direct) if os.environ.get("RS_PEER_EXCHANGE", "1") == "1" else None
    kw = dict(fused=True, device=dev, sharded=sharded, exchange=exchange)
    fm = FieldFM(cards, D, seed=1, **kw)
    ffm = FieldFFM(cards, D, seed=2, **kw)
    loss_fn = torch.nn.BCELoss()
    trainers = []
    for m in (ffm, fm):        # FFM first: the batch's sort / exchange plan (shared by both models) overlaps the long FFM forward
        opt = FusedRowOptimizer(m, torch.optim.SGD([m.bias], lr=LR), lr=LR, kind="sgd")
        trainers.append(Trainer(m, loss_fn, opt))
    return fm, ffm, trainers, loss_fn


DUMP_ROWS = 8192      # table rows sampled by --dump-outputs: 8192 x 416 floats of FFM = 13.6 MB


def c2_job(cards, B, dist_name, dev, world, rank, args, local, n_pool=8, graph=True, dump_dir=None):
    """-> (legs, n_uniq of one batch) for the FM + FFM step on `cards`.  With `dump_dir`, the outputs of the last
    timed step are written there as .npy files (see dump_c2_outputs)."""
    from deeplearningrecommendationsystem_b200 import ops
    fm, ffm, trainers, loss_fn = build_c2(cards, dev, world)
    if dump_dir is not None and fm.sharded:
        raise ValueError("--dump-outputs samples rows of unsharded tables: run it on one GPU")
    pool = [((i,), y) for i, y in (make_ids(cards, B, 1234 + rank * 100 + k, dist_name, dev) for k in range(n_pool))]

    def step(ins, y):
        for tr in trainers:
            tr.train_loop(ins[0], train_rating=y)
        return trainers[0].train_loss

    after_timed = None
    if dump_dir is not None:
        def after_timed():
            dump_c2_outputs(dump_dir, trainers, (ffm, fm), pool[(args.steps - 1) % len(pool)][0][0])

    gstep = None
    if graph and (world == 1 or os.environ.get("RS_GRAPH_SHARDED", "1") == "1"):
        from deeplearningrecommendationsystem_b200.graph import GraphedTrainStep
        gs = GraphedTrainStep(ffm, loss_fn, trainers[0].optimizer, warmup=1, also=[(fm, loss_fn, trainers[1].optimizer)])

        def gstep(ins, y):
            for tr in trainers:   # drop the eager leg's autograd graphs: their AccumulateGrad nodes are bound to its stream
                tr.predictions_train = tr.train_loss = None
            return gs(ins[0], rating=y)[1]
    legs = run_legs(step, pool, B, args, world, dev, local, graph_step=gstep, extra_warmup=3 if world > 1 else 0,
                    after_timed=after_timed)
    segs = ops.dedup_sort(pool[0][0][0], F, fm.offsets_host, fm.total_rows)
    n_uniq = segs.n_uniq
    del trainers, fm, ffm, pool
    torch.cuda.empty_cache()
    return legs, n_uniq


def dump_c2_outputs(out_dir, trainers, models, ids):
    """Write what the caller of the timed FFM + FM step holds after its last step, as float32 .npy files: each model's
    predictions (B x 1), loss and bias, and the rows of its table at DUMP_ROWS lookups of the last batch `ids` (the rows
    that step updated), picked by a fixed seed.  The inputs and the initial tables are seeded, so two builds run with the
    same arguments can be compared file by file."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    n = ids.numel()
    pick = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:DUMP_ROWS]
    offsets = torch.tensor(models[0].offsets_host, dtype=torch.int64)
    rows = (ids.reshape(-1)[pick.to(ids.device)].cpu() + offsets[pick % ids.shape[1]]).to(ids.device)
    out = {}
    for name, tr, m in zip(("ffm", "fm"), trainers, models):
        out[f"{name}_predictions"] = tr.predictions_train
        out[f"{name}_loss"] = tr.train_loss.reshape(1)
        out[f"{name}_bias"] = m.bias
        out[f"{name}_table_rows"] = m.weight[rows]
    for name, t in out.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), t.detach().float().cpu().numpy())


def c2_rooflines(legs, B, n_uniq, tag):
    """FFM bwd+update (seg_stream) and FFM forward: algorithmic bytes from this run's own unique-row count."""
    n, rb = B * F, F * D * 4
    out = {}
    k = legs["kern"]
    if "segment_update[w416]" in k:
        out["segment_update"] = hbm_roofline(
            "rs_segment_update on FFM rows (416 floats): scale gather + seg_stream_kernel<SGD> + combine",
            f"{n} lookups x {rb} B Jacobian-stash rows read + {n_uniq} unique table rows x {rb} B read and written + {n} x 20 B records/scales",
            n * rb + 2 * n_uniq * rb + n * 20, k["segment_update[w416]"], traffic=ncu_traffic(f"segment_update[w416]/{tag}"))
    if "ffm_fwd" in k:
        out["ffm_fwd"] = hbm_roofline(
            "ffm_fwd_kernel", f"{n_uniq} unique table rows x {rb} B read + {n} x {rb} B Jacobian stash written + ids",
            n_uniq * rb + n * rb + n * 8, k["ffm_fwd"], traffic=ncu_traffic(f"ffm_fwd/{tag}"))
    return out


def verify_sharded(dev, world, rank):
    """N-rank row-sharded FM + FFM steps == the 1-GPU steps on the concatenated global batch (light cardinalities, 3 steps),
    for both exchange implementations; every rank runs the sharded side, rank 0 the single-GPU side."""
    import torch.distributed as dist
    from deeplearningrecommendationsystem_b200 import dist as rsdist, ops
    from deeplearningrecommendationsystem_b200.nfield import FieldFFM, FieldFM, _xavier_concat
    from deeplearningrecommendationsystem_b200.optim import FusedRowOptimizer
    from deeplearningrecommendationsystem_b200.trainer import Trainer
    cards = [min(c, 1 << 13) for c in CRITEO]
    B, steps, lr = 2048, 3, 0.5
    ids, y = make_ids(cards, B, 99 + rank, "uniform", dev)
    all_ids = [torch.empty_like(ids) for _ in range(world)]
    all_y = [torch.empty_like(y) for _ in range(world)]
    dist.all_gather(all_ids, ids)
    dist.all_gather(all_y, y)
    out = {}
    label = {"hybrid": "small tables (< 4096 rows) replicated + rs_replica_sgd, large ones row-sharded over dist.DeviceRowExchange (the bench's placement)",
             "device": "every table row-sharded, dist.DeviceRowExchange (peer-memory kernels, no host sync)",
             "nccl": "every table row-sharded, dist.RowExchange (NCCL all_to_all_single)"}
    for name in ("hybrid", "device", "nccl"):
        progress(f"  verify: {name}")
        os.environ["RS_PEER_EXCHANGE"] = "0" if name == "nccl" else "1"
        ex = rsdist.DeviceRowExchange() if name != "nccl" else None
        errs = []
        for cls, width in ((FieldFFM, F * D), (FieldFM, D)):
            glob = _xavier_concat(cards, width, D, dev, seed=5)                  # same bits on every rank (same device type, same seed)
            m = cls(cards, D, seed=5, device=dev, sharded=True, exchange=ex, replicate_below=4096 if name == "hybrid" else 0)
            assert m.hybrid == (name == "hybrid")
            m.load_global(glob)
            tr = Trainer(m, torch.nn.BCELoss(), FusedRowOptimizer(m, torch.optim.SGD([m.bias], lr=lr), lr=lr))
            preds = []
            for _ in range(steps):
                tr.train_loop(ids, train_rating=y)
                preds.append(tr.predictions_train.detach().clone())
            sh_total = m.big_total
            rows = [(sh_total - r + world - 1) // world for r in range(world)]
            pad = torch.zeros(max(rows), width, device=dev)
            pad[: m.weight.shape[0]] = m.weight.data
            got = [torch.empty_like(pad) for _ in range(world)]
            dist.all_gather(got, pad)
            if rank == 0:
                full = m.assemble_global([got[r][: rows[r]] for r in range(world)])
                s = cls(cards, D, seed=5, device=dev)
                s.weight.data.copy_(glob)
                ts = Trainer(s, torch.nn.BCELoss(), FusedRowOptimizer(s, torch.optim.SGD([s.bias], lr=lr), lr=lr, data_parallel=False))
                gi, gy = torch.cat(all_ids), torch.cat(all_y)
                for k in range(steps):
                    ts.train_loop(gi, train_rating=gy)
                    want = ts.predictions_train.detach()[:B]
                    errs.append(float(((preds[k] - want).abs() / want.abs().clamp_min(1e-6)).max()))
                moved = (s.weight.data - glob).abs().max()
                errs.append(float((full - s.weight.data).abs().max() / moved.clamp_min(1e-12)))   # relative to the size of the update
                errs.append(float((m.bias.detach() - s.bias.detach()).abs().max() / s.bias.detach().abs().max().clamp_min(1e-12)))
                del s, ts, full
            del m, tr, glob, got, pad
            torch.cuda.empty_cache()
        ops.check_status(dev)
        if rank == 0:
            out[name] = {"max_rel_err": max(errs), "placement": label[name], "ok": max(errs) <= 1e-4}
    os.environ["RS_PEER_EXCHANGE"] = "1"
    if rank == 0:
        out["what"] = (f"{world} ranks x B={B}, 26 fields capped at 2^13 rows, {steps} SGD steps of FFM and FM: predictions (relative) and final "
                       "tables / bias (error relative to the largest update) vs the unsharded models on the concatenated batch, rank 0")
    return out


def c5_subrecord(args, dev, world, rank, local, model="MF"):
    """BASELINE.json configs[4] (the north star's own scaling config): 2 x 100 M-row tables, row-sharded when N > 1."""
    legs, B, note = c5_job(args, dev, world, rank, local, model)
    return {"metric": METRIC, "value": world * B / (legs["ms_e2e"] / 1e3), "unit": "samples/s", "n_gpus": world, "ms_per_step": legs["ms_e2e"],
            "step_api": legs["e2e_api"], "eager": {"value": world * B / (legs["ms_step"] / 1e3), "ms_per_step": legs["ms_step"]},
            "config": {"workload": WORKLOADS["c5"] + f" [{model}]", "note": note, "batch_per_gpu": B},
            "note": "value = end-to-end leg (host ids in, loss out, every step); eager = device-resident Trainer.train_loop"}


def run_c2(args):
    import torch.distributed as dist
    from deeplearningrecommendationsystem_b200 import ops
    world, rank, local = env()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    cards = [min(c, 1 << 17) for c in CRITEO] if args.light else CRITEO
    B = args.batch
    graph = args.graph
    progress(f"c2 headline: tables built, world={world}")
    legs, n_uniq = c2_job(cards, B, args.dist, dev, world, rank, args, local, graph=graph, dump_dir=args.dump_outputs)
    progress(f"c2 headline done: {legs['ms_step']:.3f} ms eager, {legs['ms_e2e']:.3f} ms e2e")
    line = base_line(args, world, B, legs, WORKLOADS["c2"],
                     {"fields": F, "dim": D, "rows": sum(cards), "ids": args.dist, "light": bool(args.light),
                      "l2": "8 distinct id batches cycled; per-step traffic (>8 GB) far exceeds the 126 MB L2",
                      "unique_rows_per_batch": n_uniq})
    if world > 1:
        line["config"]["parallelism"] = (f"dp{world}: batch split; tables under 65536 rows replicated (per-rank dense gradient, reduced + SGD + "
                                         f"re-broadcast by rs_replica_sgd over NVLink peer memory), the larger ones row-sharded (row r on rank "
                                         f"r % {world}): the FFM forward reads their rows straight from the owners' shards, gradients go "
                                         "requester's segment-reduce -> owner's buffer; no NCCL and no host sync in the step")
    tag = f"{'light' if args.light else 'full'}-{args.dist}"
    roofs = c2_rooflines(legs, B, n_uniq, tag)
    line["roofline"] = roofs.get("segment_update")
    line["roofline_ffm_fwd"] = roofs.get("ffm_fwd")
    if rank == 0 or world > 1:
        sub_args = argparse.Namespace(**vars(args))
        sub_args.steps, sub_args.warmup = max(4, args.steps // 2), max(3, args.warmup // 2)
        if not args.quick:
            # Zipf(1.05) ids beside uniform (SURVEY 8d): same tables, heavy duplicates
            other = "zipf" if args.dist == "uniform" else "uniform"
            progress(f"{other} leg")
            zl, zu = c2_job(cards, B, other, dev, world, rank, sub_args, local, graph=graph)
            zr = c2_rooflines(zl, B, zu, f"{'light' if args.light else 'full'}-{other}")
            line[other] = {"value": world * B / (zl["ms_step"] / 1e3), "ms_per_step": zl["ms_step"], "e2e": world * B / (zl["ms_e2e"] / 1e3),
                           "unique_rows_per_batch": zu, "roofline": zr.get("segment_update"), "roofline_ffm_fwd": zr.get("ffm_fwd"),
                           "kernels_ms": zl["kern"], "steps": sub_args.steps}
            if not args.light and world == 1:
                # the config the CPU arm can hold (cardinalities capped at 2^17): GPU and CPU arms on ONE stated config
                ll, lu = c2_job([min(c, 1 << 17) for c in CRITEO], B, args.dist, dev, world, rank, sub_args, local, graph=graph)
                line["light"] = {"value": B / (ll["ms_step"] / 1e3), "ms_per_step": ll["ms_step"], "e2e": B / (ll["ms_e2e"] / 1e3),
                                 "unique_rows_per_batch": lu, "rows": sum(min(c, 1 << 17) for c in CRITEO), "steps": sub_args.steps,
                                 "note": "same config as cpu_baseline.sample / the --impl reference arm"}
            progress("c5 sub-record")
            line["c5"] = c5_subrecord(sub_args, dev, world, rank, local)
            if world > 1:
                progress("sharded == single check")
                line["sharded_equals_single"] = verify_sharded(dev, world, rank)
            progress("sub-records done")
    if rank == 0:
        if world == 1 and not args.no_cpu:
            cb = time_cpu("c2", "FM+FFM", 2, 1)
            line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


# ====================================================================================================== other configs
def c5_job(args, dev, world, rank, local, model):
    from deeplearningrecommendationsystem_b200.nfield import FieldMF, FieldNeuralCF
    from deeplearningrecommendationsystem_b200.optim import FusedRowOptimizer
    from deeplearningrecommendationsystem_b200.trainer import Trainer
    rows, B = (100_000_000 if not args.light else 1_000_000), 65536
    g = torch.Generator(device=dev).manual_seed(77 + rank)
    loss_fn = torch.nn.BCELoss()
    if model == "MF":
        m = FieldMF(rows, rows, 64, seed=3, device=dev, sharded=world > 1)
        opt = FusedRowOptimizer(m, None, lr=LR)
    else:
        m = FieldNeuralCF(rows, rows, 64, [128, 64, 32, 16], seed=3, device=dev, sharded=world > 1)
        opt = FusedRowOptimizer(m, torch.optim.SGD([p for p in m.parameters() if p.requires_grad], lr=LR), lr=LR)
    pool = []
    for _ in range(8):
        u = torch.randint(0, rows, (B,), generator=g, device=dev)
        i = torch.randint(0, rows, (B,), generator=g, device=dev)
        y = (torch.rand(B, generator=g, device=dev) < 0.3).float()
        pool.append(((u, i), y if model == "MF" else y.view(-1, 1)))
    tr = Trainer(m, loss_fn, opt)

    def step(u, i, y):
        tr.train_loop(u, i, train_rating=y)
        return tr.train_loss
    gstep = None
    if args.graph and (world == 1 or os.environ.get("RS_GRAPH_SHARDED", "1") == "1"):
        from deeplearningrecommendationsystem_b200.graph import GraphedTrainStep
        gs = GraphedTrainStep(m, loss_fn, opt, warmup=1)

        def gstep(u, i, y):
            tr.predictions_train = tr.train_loss = None
            return gs(u, i, rating=y)[1]
    legs = run_legs(lambda ins, y: step(*ins, y), pool, B, args, world, dev, local,
                    graph_step=(lambda ins, y: gstep(*ins, y)) if gstep else None, extra_warmup=3 if world > 1 else 0)
    note = f"2 x {rows} rows" + (" x 2 table pairs (GMF + MLP)" if model != "MF" else "") + ", D=64, fused sparse SGD" + \
        (f", row-sharded over {world} ranks (dist.DeviceRowExchange)" if world > 1 else "")
    del tr, m, opt, pool
    torch.cuda.empty_cache()
    return legs, B, note


def eager_reference_cuda(workload, model, dev, steps=5):
    """The unmodified reference module on this GPU in eager mode (library kernels) -- the on-box number to beat
    (SURVEY 2.2 / 8d).  None when oracle/_ref was not built."""
    ref = _ref_modules()
    if ref is None:
        return None
    g = torch.Generator().manual_seed(0)
    bce = torch.nn.BCELoss()
    if workload == "c1":
        B = 87909
        ins, y = (feature_matrix_fast(g, B, 943, 1682).to(dev),), (torch.rand(B, 1, generator=g) < 0.3).float().to(dev)
        m = ref["model.deepfm"].DeepFM(943, 1682, [512, 256, 128, 1], 128).to(dev)
        opt = torch.optim.Adam(m.parameters(), lr=1e-3, weight_decay=1e-5)
    elif workload == "c4":
        B, L, items = 8192, 100, 1_000_000
        ins = (zipf_ids(items, (B, L), g, "cpu").to(dev), torch.randint(0, items, (B,), generator=g).to(dev))
        y = (torch.rand(B, 1, generator=g) < 0.3).float().to(dev)
        m = (ref["model.din"].DIN if model == "DIN" else ref["model.dien"].DIEN)(items, 64).to(dev)
        opt = torch.optim.SGD(m.parameters(), lr=0.01)
    elif workload == "c5":
        rows, B = 1_000_000, 65536
        ins = (torch.randint(0, rows, (B,), generator=g).to(dev), torch.randint(0, rows, (B,), generator=g).to(dev))
        if model == "MF":
            m, y = ref["model.mf"].MatrixFactorization(rows, rows, 64).to(dev), (torch.rand(B, generator=g) < 0.3).float().to(dev)
        else:
            m, y = ref["model.neuralcf"].NeuralCF(rows, rows, 64, [128, 64, 32, 16]).to(dev), (torch.rand(B, 1, generator=g) < 0.3).float().to(dev)
        opt = torch.optim.SGD(m.parameters(), lr=LR)
    else:
        return None
    tr = ref["trainer.trainer"].Trainer(m, bce, opt)
    for _ in range(3):
        tr.train_loop(*ins, train_rating=y)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        tr.train_loop(*ins, train_rating=y)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    return {"value": B / (ms / 1e3), "unit": "samples/s", "ms_per_step": ms,
            "what": "unmodified reference module .to('cuda'), eager torch kernels, same shapes" + (" (1 M-row tables)" if workload == "c5" else "")}


def run_other(args):
    """c1 / c3 / c4 / c5: one JSON line per model, same contract as the headline."""
    import torch.distributed as dist
    from deeplearningrecommendationsystem_b200 import model as M
    from deeplearningrecommendationsystem_b200.nfield import FieldAFM, FieldPNN
    from deeplearningrecommendationsystem_b200.optim import FusedRowOptimizer
    from deeplearningrecommendationsystem_b200.trainer import Trainer

    world, rank, local = env()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    g = torch.Generator(device=dev).manual_seed(77 + rank)
    loss_fn = torch.nn.BCELoss()
    w = args.workload
    for model in MODELS_OF[w]:
        roof, config = None, {}
        if w == "c5":
            legs, B, note = c5_job(args, dev, world, rank, local, model)
            per = 528 + 1536 if model == "MF" else 2 * (528 + 1536)
            k = legs["kern"]
            fwd_ms = k.get("fields_fwd")
            roof = hbm_roofline("whole train step (launch bound: ~10 kernels of 10-30 us)",
                                f"SURVEY 8d: {per} B/sample (rows fwd + re-read + RMW, ids) x {B}", per * B, legs["ms_e2e"],
                                note="the step is latency bound, not bandwidth bound: 65536 x 2 rows of 256 B is 34 MB per pass; "
                                     "value uses the CUDA-graph replay time")
            config = {"note": note}
        else:
            if w == "c1":
                B = 87909
                m = M.DeepFM(943, 1682, [512, 256, 128, 1], 128).to(dev)
                opt = torch.optim.Adam(m.parameters(), lr=1e-3, weight_decay=1e-5)
                gc = torch.Generator().manual_seed(5 + rank)
                pool = [((feature_matrix_fast(gc, B, 943, 1682).to(dev),), (torch.rand(B, 1, generator=gc) < 0.3).float().to(dev)) for _ in range(2)]
                config = {"note": "drop-in model.DeepFM + torch.optim.Adam(1e-3, weight_decay=1e-5) exactly as scripts/deepfm.py:52-55 builds them; "
                                  "dense-gradient tables (reference semantics)", "l2": "inputs 15.8 MB/batch, activations (B x 768 x 4 B = 270 MB) exceed L2"}
            elif w == "c3":
                cards, B = CRITEO + [64] * 13, 32768
                m = (FieldPNN(cards, 32, [256, 128, 64, 32], seed=1, device=dev, sharded=world > 1) if model == "PNN-inner"
                     else FieldAFM(cards, 32, 64, seed=2, device=dev, sharded=world > 1))
                opt = FusedRowOptimizer(m, torch.optim.SGD([p for p in m.parameters() if p.requires_grad], lr=LR), lr=LR)
                pool = [((i,), y) for i, y in (make_ids(cards, B, 900 + rank * 100 + k, args.dist, dev) for k in range(4))]
                config = {"note": "F=39, D=32, fused sparse SGD on 33.8 M rows", "ids": args.dist}
            else:
                B, L, items = 8192, 100, args.items
                m = (M.DIN if model == "DIN" else M.DIEN)(items, 64).to(dev)
                if args.dense_tables:
                    opt = torch.optim.SGD(m.parameters(), lr=0.01)
                else:
                    m.fuse_embedding_updates()
                    opt = FusedRowOptimizer(m, torch.optim.SGD([p for p in m.parameters() if p.requires_grad], lr=0.01), lr=0.01)
                pool = []
                for _ in range(4):
                    hist = zipf_ids(items, (B, L), g, dev)
                    tgt = torch.randint(0, items, (B,), generator=g, device=dev)
                    pool.append(((hist, tgt), (torch.rand(B, 1, generator=g, device=dev) < 0.3).float()))
                config = {"note": f"L=100, D=64, {items}-row item table, " + ("dense-gradient SGD (reference semantics)" if args.dense_tables
                                                                              else "fused sparse rows (model.fuse_embedding_updates() + FusedRowOptimizer)")}
            tr = Trainer(m, loss_fn, opt)

            def step(ins, y):
                tr.train_loop(*ins, train_rating=y)
                return tr.train_loss
            gstep = None
            if args.graph and w != "c1" and (world == 1 or os.environ.get("RS_GRAPH_SHARDED", "1") == "1"):
                from deeplearningrecommendationsystem_b200.graph import GraphedTrainStep
                gs = GraphedTrainStep(m, loss_fn, opt, warmup=1)

                def gstep(ins, y):
                    tr.predictions_train = tr.train_loss = None
                    return gs(*ins, rating=y)[1]
            legs = run_legs(step, pool, B, args, world, dev, local, graph_step=gstep, extra_warmup=3 if world > 1 else 0)
            k = legs["kern"]
            if w == "c1":
                # the embedding backward of the two id tables is the largest of this package's kernels in the C1 step
                if "segment_update[w128]" in k:
                    roof = hbm_roofline("rs_segment_update[w128] (deterministic embedding backward of the user / item tables: 2 x B gradient rows "
                                        "of 128 floats segment-reduced into dense gradients)",
                                        f"2 x {B} x 512 B gradient rows read + (943 + 1682) x 512 B dense gradient written + 2 x {B} x 16 B records",
                                        2 * B * 512 + (943 + 1682) * 512 + 2 * B * 16, k["segment_update[w128]"],
                                        note="the C1 step itself is dominated by the cuBLAS fp32 towers (768->512->256->128->1) and the dense "
                                             "torch Adam sweep, scoped out by SURVEY 2.2: this package's kernels account for ~0.3 of its ~8.9 ms")
            elif w == "c3" and model == "PNN-inner":
                if "fields_fwd" in k:
                    roof = hbm_roofline("fields_fwd_kernel (39-field gather + 741 inner products + concat)",
                                        "SURVEY 8d: 4992 B rows + 312 B ids + 2964 B products + 4992 B concat per sample", (4992 + 312 + 2964 + 4992) * B, k["fields_fwd"])
            elif w == "c3":
                NP, A = 39 * 38 // 2, 64
                if "afm_fwd" in k:
                    roof = tensor_roofline("afm_fwd_tc_kernel (pair products -> P W on tcgen05, 3xTF32)", f"{B} x {NP} pairs x 2 x 32 x {A} (projection only)",
                                           B * NP * 2 * 32 * A, k["afm_fwd"])
                if "afm_bwd_tc" in k:
                    config["roofline_bwd"] = tensor_roofline("afm_bwd_chain_tc + afm_de + afm_dw_tc", f"{B} x {NP} pairs x 3 GEMMs x 2 x 32 x {A}",
                                                             3 * B * NP * 2 * 32 * A, k["afm_bwd_tc"])
            else:
                H1, H2 = (128, 64) if model == "DIN" else (64, 32)
                fl = B * L * 2 * (64 * H1 + H1 * H2)
                if "din_fwd_tc" in k:
                    roof = tensor_roofline("din_tbias + din_score_tc_kernel + din_softmax_pool (attention unit on tcgen05, 3xTF32)",
                                           f"{B} x {L} rows x 2 x (64 x {H1} + {H1} x {H2}) (concat-free first layer)", fl, k["din_fwd_tc"])
                if "din_bwd_tc" in k:
                    config["roofline_bwd"] = tensor_roofline("din_bwd_tc_kernel (data-gradient chain)", "same two GEMMs, transposed", fl, k["din_bwd_tc"])
            del tr, m, opt, pool
            torch.cuda.empty_cache()
        line = base_line(args, world, B, legs, WORKLOADS[w] + f" [{model}]", config)
        line["roofline"] = roof
        if rank == 0:
            if world == 1 and not args.no_cpu:
                try:
                    cb = time_cpu(w, model, 2, 1)
                    line["cpu_baseline"] = {k_: cb[k_] for k_ in ("value", "unit", "cores", "kind", "sample")}
                except Exception as e:      # noqa: BLE001
                    line["cpu_baseline"] = {"unavailable": str(e)}
                try:
                    line["eager_reference_cuda"] = eager_reference_cuda(w, model, dev)
                except Exception as e:      # noqa: BLE001
                    line["eager_reference_cuda"] = {"unavailable": str(e)[:200]}
            print(json.dumps(line), flush=True)
        torch.cuda.empty_cache()
    if world > 1:
        dist.destroy_process_group()


def run_rank(args):
    """SURVEY.md 8(f).1 -- catalogue ranking (`recommendation()`), one JSON line per case.  Not the headline metric.

    mf:      fused rs_mf_rank over a (users x items) catalogue vs cuBLAS matmul + torch.topk (library route) and the
             numpy oracle on the host (bounded sample of users).
    deepfm:  DeepFM.recommendation(943, frame, 1682) -- the scripts' call (scripts/deepfm.py:67) -- wall clock including
             the host-side grouping of the frame, vs the reference's one-forward-per-user loop on a sample of users."""
    import numpy as np
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from helpers import catalogue_frame
    from oracle import ranking as R
    from deeplearningrecommendationsystem_b200 import model as M, ops
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    g = torch.Generator().manual_seed(5)

    def dev_ms(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / steps

    for nu, ni, W, k, tag in ((943, 1682, 64, 1682, "ML-100k full ranking (scripts/mf.py:81)"),
                              (65536, 16384, 64, 100, "synthetic 65536 users x 16384 items, top-100")):
        U = (torch.randn(nu, W, generator=g) * 0.3).to(dev)
        V = (torch.randn(ni, W, generator=g) * 0.3).to(dev)
        ms = dev_ms(lambda: ops.mf_rank(U, V, k, check=False), args.steps, max(args.warmup, 3))
        ms_lib = dev_ms(lambda: torch.topk(U @ V.T, k, dim=1), max(args.steps // 4, 2), 2)
        ns = min(nu, 256)
        Un, Vn = U[:ns].cpu().numpy(), V.cpu().numpy()
        t0 = time.perf_counter()
        sc = (Un @ Vn.T).astype(np.float32)
        for u in range(ns):
            R.rank_desc(sc[u], k)
        cpu = ns / (time.perf_counter() - t0)
        print(json.dumps({"metric": "ranked users/sec", "value": nu / (ms / 1e3), "unit": "users/s", "n_gpus": 1, "steps": args.steps,
                          "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "vs_baseline": None, "dtype": "f32",
                          "data": "synthetic", "config": {"workload": f"rank/mf: {tag}", "users": nu, "items": ni, "width": W, "k": k},
                          "library_route_ms": ms_lib, "gpu_launches": args.steps,
                          "cpu_baseline": {"value": cpu, "unit": "users/s", "cores": 1, "kind": "port", "sample": f"{ns} users, numpy"}}))

    nu, ni = 943, 1682
    torch.manual_seed(0)
    m = M.DeepFM(nu, ni, [256, 128, 1], 128).to(dev).eval()          # scripts/deepfm.py:52
    df = catalogue_frame(g, nu, ni, shuffle=False)
    m.recommendation(32, df[df["user_id"] < 32], ni)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = m.recommendation(nu, df, ni)
    torch.cuda.synchronize()
    sec = time.perf_counter() - t0
    ns = 24
    t0 = time.perf_counter()
    with torch.no_grad():
        for u in range(ns):                                            # the reference's loop, model/deepfm.py:85-95, on this GPU
            rows = torch.Tensor(df[df["user_id"] == u].values).to(dev)
            torch.topk(m(rows), ni, dim=0).indices.view(1, -1).tolist()[0]
    loop = ns / (time.perf_counter() - t0)
    print(json.dumps({"metric": "ranked users/sec", "value": nu / sec, "unit": "users/s", "n_gpus": 1, "steps": 1, "warmup": 1,
                      "ms_per_step": sec * 1e3, "higher_is_better": True, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                      "config": {"workload": "rank/deepfm: DeepFM.recommendation(943, user_item, 1682), wall clock incl. host grouping",
                                 "rows": int(len(df)), "shape": list(out.shape)},
                      "per_user_loop_users_per_s": loop, "per_user_loop_sample": f"{ns} users, same GPU, reference control flow"}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--dist", default="uniform", choices=["uniform", "zipf"])
    ap.add_argument("--batch", type=int, default=BATCH)
    ap.add_argument("--light", action="store_true", help="cap every cardinality at 2^17 rows (fits any GPU)")
    ap.add_argument("--quick", action="store_true", help="c2 only: skip the zipf / light / c5 / verification sub-records")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--items", type=int, default=1_000_000, help="c4: rows of the item table (SURVEY 8d also names 10 M)")
    ap.add_argument("--dense-tables", action="store_true", help="c4: reference dense-gradient tables instead of fused sparse rows")
    ap.add_argument("--graph", dest="graph", action="store_true", default=True,
                    help="end-to-end leg replays the step as a CUDA graph (default; the sharded step has no host sync either)")
    ap.add_argument("--no-graph", dest="graph", action="store_false", help="eager Trainer.train_loop in the end-to-end leg too")
    ap.add_argument("--workload", default="c2", choices=["c2", "c1", "c3", "c4", "c5", "rank"],
                    help="c2 = headline (BASELINE.json configs[1]); c1/c3/c4/c5 = the other configs, one line per model")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="c2, one GPU: write the outputs of the last timed step (predictions, losses, biases, a fixed sample of "
                         "updated table rows) to DIR/<name>.npy as float32")
    args = ap.parse_args()
    if args.dump_outputs is not None and (args.impl != "b200" or args.workload != "c2"):
        ap.error("--dump-outputs covers the c2 workload of the GPU implementation")
    if args.impl == "reference":
        if args.workload == "rank":
            args.workload = "c2"
        run_reference(args)
    elif args.workload == "c2":
        run_c2(args)
    elif args.workload == "rank":
        run_rank(args)
    else:
        run_other(args)


if __name__ == "__main__":
    main()
