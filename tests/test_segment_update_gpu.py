"""rs_segment_update -- the sort / segment-reduce fused with the row update -- on every dispatch leaf, in all three modes
(RS_UPD_GRAD, SGD, lazy Adam), against float64; and the one-step-per-opt.step() rule of FusedRowOptimizer.

The dispatch of rs_segment_update (segment.cu: use_stream, dispatch_update; segment_stream.cu: launch_seg_stream,
launch_na) is restated in python below and checked against the source text; the GPU cases are drawn from that
restatement and a CPU test asserts that every reachable leaf has one.

Bars, from float64 sums of the fp32 per-lookup gradients (S = segment sum of |terms|, eps32 = 2^-24):
  GRAD  |g_gpu - g64| <= 1e-5 |g64| + 4 eps32 S
  SGD   |w_gpu - w64| <= 1e-6 |w64| + lr (1e-5 |g64| + 4 eps32 S)      (g64 includes wd w)
  Adam  m, v: the float64 recurrences driven by the GPU's previous m / v, with the gradient bound propagated through them;
        w: float64 Adam on the GPU's own new m, v and previous w, to 4 eps32 |w| + 8 eps32 step_size |m / denom| -- a few
        ulp, so a wrong bias correction, decay term, eps or step count fails outright.  Secondary: DESIGN.md's free-running
        rule over the three steps (>= 99 % within 1e-5, none beyond steps lr).
Untouched rows (and their m, v) stay bit-identical; every streaming case is run twice and must repeat bit for bit.
"""
import copy
import os
import re

import numpy as np
import pytest
import torch

from oracle import optim as ooptim

EPS32 = 2.0 ** -24
SMEM = 232448                       # shared memory per SM on B200 (227 KB)
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "deeplearningrecommendationsystem_b200", "csrc")
F32 = lambda x: float(np.float32(x))   # noqa: E731  the kernels take lr, wd, betas, eps as float
B1, B2, EPS = F32(0.9), F32(0.999), F32(1e-8)
SGD_LR, ADAM_LR, WDS, ADAM_STEPS = F32(0.05), F32(1e-2), (0.0, F32(1e-2)), 3
SEG_LENS = (1, 63, 64, 65, 127, 128, 129, 512, 513)     # around RS_CHUNK = 64 and the RS_UNIT = 512 work units

# ============================================================================ dispatch restatement
LANE4 = ((1, 1, 1), (2, 2, 1), (4, 4, 1), (8, 8, 1), (16, 16, 1), (32, 32, 1), (64, 32, 2), (128, 32, 4), (256, 32, 8))
LANE4_LAST = (32, 16)                # (GS, NA) above the last bound of W / 4
LANE1 = ((1, 1, 1), (32, 32, 1), (128, 32, 4), (512, 32, 16))   # (W <= bound, GS, NA) for W not a multiple of 4
NCT, SR, MAX_ST, STATIC = 128, 8, 12, 6 * 1024
SOURCES = ("dense", "stash", "stash*scalar", "stash*vector", "stash+dense")


def use_stream(W, src, no_stream=False):
    """segment.cu: wide rows with one gradient source and at most a per-sample scalar scale take the streaming kernel"""
    return W % 4 == 0 and 96 <= W <= 640 and src not in ("stash+dense", "stash*vector") and not no_stream


def stream_leaf(W, ctas1=False, half_sm=False):
    """launch_seg_stream + launch_na (no routes): ((kernel, NA, CTAs per SM, BATCH), ring stages) or (None, 0)"""
    wv = W // 4
    NA = 1 if wv <= NCT else (2 if wv <= 2 * NCT else 4)
    stage = 2 * SR * W * 4
    per_sm = 1 if ctas1 else 2
    small = per_sm == 2
    nst = 0
    if per_sm == 2:
        nst = (SMEM // 2 - STATIC - 1024) // stage
        if nst < 3:
            per_sm, small = 1, False
        elif half_sm:
            per_sm = 1
    if not small:
        nst = (200 * 1024) // stage
    nst = min(nst, MAX_ST)
    if nst < (3 if small else 5):
        return None, 0
    return ("stream", NA, per_sm, 2 if small else 4), nst


def route(W, src="dense", no_stream=False, ctas1=False, half_sm=False):
    """rs_segment_update's chunk-pass kernel for rows of W floats: ((kind, ...), stages) or (None, 0) = refused before any
    launch (width > 2048, or not a multiple of 4 and > 512)"""
    if not 1 <= W <= 2048:
        return None, 0
    if use_stream(W, src, no_stream):
        return stream_leaf(W, ctas1, half_sm)
    if W % 4 == 0:
        for bound, GS, NA in LANE4:
            if W // 4 <= bound:
                return ("lane", 4, GS, NA), 0
        return ("lane", 4) + LANE4_LAST, 0
    for bound, GS, NA in LANE1:
        if W <= bound:
            return ("lane", 1, GS, NA), 0
    return None, 0


def knobs_of(env):
    return dict(no_stream="RS_NO_STREAM" in env, ctas1=env.get("RS_SEG_CTAS") == "1")


# (W, gradient source, environment, half_sm): one or more per leaf
LEAF_CASES = [
    (4, "dense", {}, False), (8, "dense", {}, False), (16, "dense", {}, False), (32, "dense", {}, False),
    (64, "dense", {}, False), (88, "dense", {}, False),
    (256, "stash+dense", {}, False), (416, "dense", {"RS_NO_STREAM": "1"}, False),
    (768, "dense", {}, False), (1024, "dense", {}, False), (1248, "dense", {}, False), (2048, "dense", {}, False),
    (1, "dense", {}, False), (10, "dense", {}, False), (90, "dense", {}, False), (510, "dense", {}, False),
    (96, "dense", {}, False), (416, "dense", {}, False), (512, "dense", {}, False),
    (416, "dense", {"RS_SEG_CTAS": "1"}, False), (416, "dense", {}, True),
    (528, "dense", {}, False), (640, "dense", {}, False), (528, "dense", {}, True),
]
REFUSED = (514, 2052)


def case_id(c):
    W, src, env, half = c
    leaf, nst = route(W, src, half_sm=half, **knobs_of(env))
    tag = "-".join(str(x) for x in leaf) + (f"x{nst}" if nst else "")
    return f"W{W}-{src}-{tag}" + "".join(f"-{k}" for k in env) + ("-half_sm" if half else "")


def test_dispatch_restatement_tracks_the_sources():
    """the restatement above against segment.cu / segment_stream.cu, and every reachable leaf covered by LEAF_CASES"""
    def norm(name):
        with open(os.path.join(CSRC, name)) as f:
            return re.sub(r"\s+", " ", f.read())
    seg, stm = norm("segment.cu"), norm("segment_stream.cu")
    assert ("P.use_stream = (W % 4 == 0 && W >= 96 && W <= 640 && !(u->stash && u->dense) && (!u->scale || u->scale_width == 1) "
            "&& !getenv(\"RS_NO_STREAM\")) ? 1 : 0;") in seg
    assert "u->width >= 1 && u->width <= 2048" in seg
    assert "rs_segment_update: width %d not a multiple of 4 and > 512" in seg
    lane4 = [tuple(int(x) for x in m) for m in re.findall(r"if \(wv <= (\d+)\) return launch_mode<4, (\d+), (\d+)>", seg)]
    assert lane4 == list(LANE4)
    assert "return launch_mode<4, %d, %d>(P, mode, n, st); }" % LANE4_LAST in seg
    lane1 = re.findall(r"if \(W (==|<=) (\d+)\) return launch_mode<1, (\d+), (\d+)>", seg)
    assert [tuple(int(x) for x in m[1:]) for m in lane1] == list(LANE1)
    # launch_seg_stream: NA by W / 4 against NCT consumer threads
    assert "constexpr int SR = 8;" in stm and "constexpr int NCW = 4;" in stm and "constexpr int NCT = NCW * 32;" in stm
    assert "constexpr int MAX_ST = 12;" in stm
    assert ("if (wv <= NCT) return launch_na<1>(P, (int)n, mode, st); if (wv <= 2 * NCT) return launch_na<2>(P, (int)n, mode, st); "
            "return launch_na<4>(P, (int)n, mode, st);") in stm
    # launch_na: CTAs per SM, ring stages, BATCH
    for s in ("const size_t stage_bytes = (size_t)2 * SR * P.W * 4;", "const size_t static_bytes = 6 * 1024;",
              "int per_sm = (out_slots == 0) ? 2 : 1;", "per_sm = (atoi(e) == 1) ? 1 : per_sm;", "bool small_ring = per_sm == 2;",
              "nst = (int)((232448 / 2 - static_bytes - 1024) / stage_bytes);", "if (nst < 3) per_sm = 1, small_ring = false;",
              "else if (P.half_sm) per_sm = 1;", "if (!small_ring) nst = (int)((200 * 1024 - out_bytes) / stage_bytes);",
              "if (nst > MAX_ST) nst = MAX_ST;", "if (nst < (small_ring ? 3 : 5)) {",
              "if (small_ring) RS_LAUNCH_STREAM(M, PUSH, 2); else RS_LAUNCH_STREAM(M, PUSH, 4);"):
        assert s in stm, s
    # grid-stride caps of the chunk and combine passes (the thresholds of the grid-stride cases below)
    assert "int cap = rs::num_sms() * 64;" in seg
    assert "int cblocks = (int)(cblocks64 < rs::num_sms() * 8 ? cblocks64 : rs::num_sms() * 8);" in seg

    reachable = set()
    for W in range(1, 2049):
        for src in SOURCES:
            for env in ({}, {"RS_NO_STREAM": "1"}, {"RS_SEG_CTAS": "1"}):
                for half in (False, True):
                    leaf, nst = route(W, src, half_sm=half, **knobs_of(env))
                    if leaf is not None:
                        reachable.add(leaf)
                    if use_stream(W, src, knobs_of(env)["no_stream"]):
                        assert leaf is not None, W          # the streaming kernel refuses nothing use_stream sends it
    # use_stream caps W at 640 (W / 4 <= 160 <= 2 NCT): launch_seg_stream's NA = 4 branch is never taken
    assert not any(leaf[0] == "stream" and leaf[1] == 4 for leaf in reachable)
    assert route(416)[0] == ("stream", 1, 2, 2) and route(416)[1] == 4
    assert route(96)[1] == 12 and route(512)[1] == 3 and route(528) == (("stream", 2, 2, 2), 3) and route(640) == (("stream", 2, 1, 4), 5)
    assert route(416, ctas1=True) == (("stream", 1, 1, 4), 7) and route(416, half_sm=True) == (("stream", 1, 1, 2), 4)
    covered = {route(W, src, half_sm=half, **knobs_of(env))[0] for W, src, env, half in LEAF_CASES}
    assert None not in covered
    assert covered == reachable, sorted(map(str, reachable - covered))
    for W in REFUSED:
        assert route(W)[0] is None


def test_adam_rows_with_weight_decay_equals_torch_adam():
    """oracle.optim.adam_rows(wd) is torch.optim.Adam(weight_decay=wd) where every row is touched (lazy = dense there)"""
    g = torch.Generator().manual_seed(0)
    R, W = 50, 8
    p0 = torch.randn(R, W, generator=g, dtype=torch.float64)
    ids = torch.cat([torch.arange(R), torch.randint(0, R, (300,), generator=g)])
    ref = torch.nn.Parameter(p0.clone())
    opt = torch.optim.Adam([ref], lr=1e-2, weight_decay=1e-2)
    t, m, v = p0.clone(), torch.zeros_like(p0), torch.zeros_like(p0)
    for step in (1, 2, 3):
        G = torch.randn(ids.numel(), W, generator=g, dtype=torch.float64)
        ref.grad = torch.zeros(R, W, dtype=torch.float64).index_add_(0, ids, G)
        opt.step()
        ooptim.adam_rows(t, m, v, ids, G, step, lr=1e-2, wd=1e-2)
        st = opt.state[ref]
        np.testing.assert_allclose(m.numpy(), st["exp_avg"].numpy(), rtol=1e-12, atol=1e-15)
        np.testing.assert_allclose(v.numpy(), st["exp_avg_sq"].numpy(), rtol=1e-12, atol=1e-15)
        np.testing.assert_allclose(t.numpy(), ref.data.numpy(), rtol=1e-12, atol=1e-15)


# ============================================================================ GPU: data and float64 references
def _ops():
    from deeplearningrecommendationsystem_b200 import ops
    return ops


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


WORST = {}


@pytest.fixture(scope="module", autouse=True)
def report_worst():
    yield
    if WORST:
        print("\n[segment-update] worst error / bound: " + ", ".join(f"{k} {v:.3f}" for k, v in sorted(WORST.items())))


def _note(what, ratio):
    WORST[what] = max(WORST.get(what, 0.0), ratio)


def _col(g, n, rows, specials=True, hot=0, lo=10, hi=None):
    """n local ids of one field: rows 0..8 with the lengths SEG_LENS, row 9 with `hot` lookups, the rest uniform over
    [lo, hi) (rows at and above hi are never looked up), in random order"""
    parts = []
    if specials:
        parts += [torch.full((c,), r, dtype=torch.int64) for r, c in enumerate(SEG_LENS)]
    if hot:
        parts.append(torch.full((hot,), 9, dtype=torch.int64))
    k = n - sum(p.numel() for p in parts)
    assert k >= 0
    parts.append(torch.randint(lo, hi if hi is not None else rows, (k,), generator=g))
    col = torch.cat(parts)
    return col[torch.randperm(n, generator=g)]


class Case:
    """lookups (B, F) with row offsets, the fp32 gradient sources and their float64 per-lookup gradient"""

    def __init__(self, W, src, F=1, seed=0, n=48000, ids=None, cards=None, n_valid=None):
        g = torch.Generator().manual_seed(seed)
        if ids is None:
            if F == 1:
                cards = [3000]
                ids = _col(g, n, 3000, hot=20000, hi=2900).view(-1, 1)        # row 9 takes 42 % of the lookups
            else:
                assert F == 3
                cards, B = [50, 4000, 700], n // 3
                ids = torch.stack([torch.randint(0, 50, (B,), generator=g), _col(g, B, 4000, hot=6000, hi=3900),
                                   (torch.rand(B, generator=g) ** 3 * 650).long()], dim=1)
        self.W, self.src, self.F, self.cards = W, src, ids.shape[1], cards
        self.offs = [sum(cards[:k]) for k in range(len(cards))]
        self.total = sum(cards)
        self.B, self.n = ids.shape[0], ids.numel()
        self.ids = ids.cuda()
        keys = (ids + torch.tensor(self.offs)).reshape(-1).cuda()
        nv = self.n if n_valid is None else n_valid
        self.nv = nv
        gd = torch.Generator(device="cuda").manual_seed(seed + 1)
        rnd = lambda *s: torch.randn(*s, generator=gd, device="cuda")     # noqa: E731
        self.stash = self.scale = self.dense = None
        G64 = torch.zeros(self.B, self.F, W, dtype=torch.float64, device="cuda")
        A64 = torch.zeros_like(G64)
        if src != "dense":
            self.stash = rnd(self.B, self.F, W) * 0.01
            t = self.stash.double()
            if src == "stash*scalar":
                self.scale = rnd(self.B)
                t = t * self.scale.double()[:, None, None]
            elif src == "stash*vector":
                self.scale = rnd(self.B, W)
                t = t * self.scale.double()[:, None, :]
            G64 += t
            A64 += t.abs()
        if src in ("dense", "stash+dense"):
            self.dense = rnd(self.B, self.F, W) * 0.01
            G64 += self.dense.double()
            A64 += self.dense.double().abs()
        G64, A64, keys = G64.view(-1, W)[:nv], A64.view(-1, W)[:nv], keys[:nv]
        self.uniq, inv = torch.unique(keys, return_inverse=True)
        nu = self.uniq.numel()
        self.gsum = torch.zeros(nu, W, dtype=torch.float64, device="cuda").index_add_(0, inv, G64)
        self.S = torch.zeros(nu, W, dtype=torch.float64, device="cuda").index_add_(0, inv, A64)
        self.counts = torch.bincount(inv, minlength=nu)
        mask = torch.ones(self.total, dtype=torch.bool, device="cuda")
        mask[self.uniq] = False
        self.untouched = mask.nonzero().view(-1)
        self.table0 = torch.randn(self.total, W, generator=gd, device="cuda")
        self.m0 = rnd(self.total, W) * 0.01
        self.v0 = torch.rand(self.total, W, generator=gd, device="cuda") * 1e-4

    def sources(self):
        return dict(stash=self.stash, scale=self.scale, dense=self.dense)

    def sort(self, n_valid=None):
        return _ops().dedup_sort(self.ids, self.F, self.offs, self.total, max_width=self.W, reuse_workspace=False, n_valid=n_valid)


def _check(got, want, bound, what):
    err = (got.double() - want).abs()
    bad = err > bound
    if bool(bad.any()):
        r, e = (int(x) for x in bad.nonzero()[0])
        raise AssertionError(f"{what}: {int(bad.sum())} elements outside the bound; first at touched row {r}, element {e}: "
                             f"gpu {float(got[r, e])!r} want {float(want[r, e])!r} bound {float(bound[r, e]):.3e}")
    ratio = float((err / bound.clamp_min(1e-300)).max())
    mode = what.split(":")[0]
    _note(mode + (" " + what.split()[-1] if mode == "adam" else ""), ratio)
    return ratio


def _same_bits(a, b, what):
    assert torch.equal(a.view(torch.int32), b.view(torch.int32)), what


def run_modes(c, segs, label, env=(), half_sm=False):
    """GRAD, SGD (wd 0, 1e-2) and three Adam steps (wd 0, 1e-2) on one case; returns every final output for the bit
    comparisons of the callers"""
    ops = _ops()
    W, F, U = c.W, c.F, c.uniq
    out = {}
    # ---- GRAD: rows are written, not accumulated; untouched rows keep their (random) contents
    dg = c.m0.clone()
    ops.segment_update(segs, ops.RS_UPD_GRAD, W, F, dense_grad=dg, half_sm=half_sm, **c.sources())
    _check(dg[U], c.gsum, 1e-5 * c.gsum.abs() + 4 * EPS32 * c.S, f"grad: {label}")
    _same_bits(dg[c.untouched], c.m0[c.untouched], f"grad {label}: untouched rows")
    out["grad"] = dg
    for wd in WDS:
        # ---- SGD
        t = c.table0.clone()
        ops.segment_update(segs, ops.RS_UPD_SGD, W, F, table=t, lr=SGD_LR, wd=wd, half_sm=half_sm, **c.sources())
        w0 = c.table0[U].double()
        g = c.gsum + wd * w0
        w64 = w0 - SGD_LR * g
        _check(t[U], w64, 1e-6 * w64.abs() + SGD_LR * (1e-5 * g.abs() + 4 * EPS32 * (c.S + wd * w0.abs())), f"sgd: {label} wd={wd}")
        _same_bits(t[c.untouched], c.table0[c.untouched], f"sgd {label}: untouched rows")
        out[f"sgd{wd}"] = t
        # ---- Adam, three steps on the same summed gradient
        t, m, v = c.table0.clone(), c.m0.clone(), c.v0.clone()
        fw, fm, fv = c.table0[U].double(), c.m0[U].double(), c.v0[U].double()      # free-running float64 trajectory
        for step in range(1, ADAM_STEPS + 1):
            wp, mp, vp = t[U].double(), m[U].double(), v[U].double()
            ops.segment_update(segs, ops.RS_UPD_ADAM, W, F, table=t, m=m, v=v, lr=ADAM_LR, wd=wd, betas=(B1, B2), eps=EPS, step=step,
                               half_sm=half_sm, **c.sources())
            what = f"adam: {label} wd={wd} step {step}"
            g = c.gsum + wd * wp
            eg = 1e-5 * g.abs() + 4 * EPS32 * (c.S + wd * wp.abs()) + 2 * EPS32 * g.abs()
            m64 = mp + (1 - B1) * (g - mp)
            v64 = B2 * vp + (1 - B2) * g * g
            _check(m[U], m64, (1 - B1) * eg + 4 * EPS32 * (mp.abs() + m64.abs() + (1 - B1) * g.abs()), what + " m")
            _check(v[U], v64, (1 - B2) * (2 * g.abs() * eg + eg * eg) + 4 * EPS32 * (B2 * vp + v64 + (1 - B2) * g * g) + 1e-45,
                   what + " v")
            bc1, bc2 = 1 - B1 ** step, 1 - B2 ** step
            step_size = ADAM_LR / bc1
            mg, vg = m[U].double(), v[U].double()
            q = mg / (vg.sqrt() / np.sqrt(bc2) + EPS)
            w64 = wp - step_size * q
            _check(t[U], w64, 4 * EPS32 * w64.abs() + 8 * EPS32 * step_size * q.abs() + 1e-45, what + " w")
            gf = c.gsum + wd * fw
            fm = fm + (1 - B1) * (gf - fm)
            fv = B2 * fv + (1 - B2) * gf * gf
            fw = fw - step_size * fm / (fv.sqrt() / np.sqrt(bc2) + EPS)
        dev = (t[U].double() - fw).abs()
        assert float((dev <= 1e-5).double().mean()) >= 0.99 and float(dev.max()) <= ADAM_STEPS * ADAM_LR, \
            f"adam {label} wd={wd}: free-running trajectory, {float((dev <= 1e-5).double().mean()):.4f} within 1e-5, max {float(dev.max()):.3e}"
        for a, a0, name in ((t, c.table0, "w"), (m, c.m0, "m"), (v, c.v0, "v")):
            _same_bits(a[c.untouched], a0[c.untouched], f"adam {label} wd={wd}: untouched rows of {name}")
        out[f"adam{wd}"] = (t, m, v)
    ops.check_status()
    return out


def _same_outputs(a, b, what):
    for k in a:
        for x, y in zip(*((a[k], b[k]) if isinstance(a[k], tuple) else ((a[k],), (b[k],)))):
            _same_bits(x, y, f"{what}: {k}")


# ============================================================================ GPU: the kernel matrix
@pytest.mark.gpu
@pytest.mark.parametrize("case", LEAF_CASES, ids=case_id)
def test_every_dispatch_leaf_in_all_modes(case, monkeypatch):
    """segments of 1..513 lookups, a row with 42 % of them (combine groups of several chunks at every GS), all three
    modes, wd 0 and 1e-2; streaming leaves twice, bit-identical"""
    W, src, env, half = case
    for k, val in env.items():
        monkeypatch.setenv(k, val)
    leaf, _ = route(W, src, half_sm=half, **knobs_of(env))
    c = Case(W, src, F=1, seed=W)
    assert sorted(set(SEG_LENS) - set(c.counts.tolist())) == [] and int(c.counts.max()) >= 0.4 * c.n
    segs = c.sort()
    out = run_modes(c, segs, case_id(case), half_sm=half)
    if leaf[0] == "stream":
        _same_outputs(out, run_modes(c, segs, case_id(case), half_sm=half), f"{case_id(case)} second run")


@pytest.mark.gpu
@pytest.mark.parametrize("src", SOURCES)
@pytest.mark.parametrize("W", [88, 416])
def test_gradient_sources_with_row_offsets(W, src):
    """every gradient source at a lane-group width and a streaming width, F = 3 fields with row offsets; the per-sample
    scale is indexed by lookup / F"""
    c = Case(W, src, F=3, seed=7 * W + SOURCES.index(src))
    assert sorted(set(SEG_LENS) - set(c.counts.tolist())) == []
    segs = c.sort()
    leaf, _ = route(W, src)
    out = run_modes(c, segs, f"W{W} F3 {src}")
    if leaf[0] == "stream":
        _same_outputs(out, run_modes(c, segs, f"W{W} F3 {src}"), f"W{W} {src} second run")


@pytest.mark.gpu
@pytest.mark.parametrize("src", ["dense", "stash*scalar"])
@pytest.mark.parametrize("W", [416, 512])
def test_lane_group_and_streaming_kernels_agree_bit_for_bit(W, src, monkeypatch):
    """both kernels add a chunk's rows in ascending position with the scale multiply and the add rounded separately, so
    GRAD and SGD agree to the bit; for Adam the agreement is reported, not required"""
    ops = _ops()
    c = Case(W, src, F=3, seed=W + 1)
    segs = c.sort()
    outs = []
    for no_stream in (False, True):
        if no_stream:
            monkeypatch.setenv("RS_NO_STREAM", "1")
        assert route(W, src, no_stream=no_stream)[0][0] == ("lane" if no_stream else "stream")
        r = {}
        r["grad"] = torch.zeros(c.total, W, device="cuda")
        ops.segment_update(segs, ops.RS_UPD_GRAD, W, c.F, dense_grad=r["grad"], **c.sources())
        for wd in WDS:
            r[f"sgd{wd}"] = c.table0.clone()
            ops.segment_update(segs, ops.RS_UPD_SGD, W, c.F, table=r[f"sgd{wd}"], lr=SGD_LR, wd=wd, **c.sources())
        t, m, v = c.table0.clone(), c.m0.clone(), c.v0.clone()
        ops.segment_update(segs, ops.RS_UPD_ADAM, W, c.F, table=t, m=m, v=v, lr=ADAM_LR, wd=WDS[1], betas=(B1, B2), eps=EPS, step=1,
                           **c.sources())
        r["adam"] = (t, m, v)
        outs.append(r)
    for k in ("grad",) + tuple(f"sgd{wd}" for wd in WDS):
        _same_bits(outs[0][k], outs[1][k], f"W{W} {src} {k}: streaming vs lane-group")
    same = [torch.equal(a, b) for a, b in zip(outs[0]["adam"], outs[1]["adam"])]
    print(f"\n[segment-update] W{W} {src}: Adam streaming vs lane-group bit-identical (w, m, v): {same}")


@pytest.mark.gpu
def test_combine_grid_stride_over_multi_chunk_segments():
    """more multi-chunk segments than the combine pass has CTAs (SMs * 8): every CTA loops"""
    sms = _sms()
    rows = sms * 8 + 150
    g = torch.Generator().manual_seed(5)
    ids = torch.arange(rows).repeat_interleave(70)
    ids = ids[torch.randperm(ids.numel(), generator=g)].view(-1, 1)
    c = Case(8, "dense", ids=ids, cards=[rows + 20], seed=5)
    assert int((c.counts > 64).sum()) > sms * 8
    run_modes(c, c.sort(), "combine grid-stride W8")


@pytest.mark.gpu
def test_chunk_grid_stride_over_many_chunks():
    """more chunks than the chunk pass's capped grid covers at once (SMs * 64 CTAs of 8 lane groups at W = 88)"""
    sms = _sms()
    rows = sms * 64 * 8 + 30000
    g = torch.Generator().manual_seed(6)
    ids = torch.cat([torch.arange(rows), torch.randint(0, rows, (20000,), generator=g)])
    ids = ids[torch.randperm(ids.numel(), generator=g)].view(-1, 1)
    c = Case(88, "dense", ids=ids, cards=[rows + 100], seed=6)
    assert c.uniq.numel() > sms * 64 * 8
    run_modes(c, c.sort(), "chunk grid-stride W88")


@pytest.mark.gpu
@pytest.mark.parametrize("W", [88, 416])
def test_padded_sort_updates_only_the_valid_prefix(W):
    """the row-sharded owner update: a receive list of fixed capacity whose fill level is a device scalar (n_valid).
    Padding ids point at rows no real lookup touches; those rows and their m, v stay bit-identical."""
    g = torch.Generator().manual_seed(W)
    n, nv, rows = 9000, 7000, 3000
    ids = _col(g, n, rows, hot=2000, hi=2800).view(-1, 1)
    ids[nv:] = torch.randint(2900, rows, (n - nv, 1), generator=g)
    c = Case(W, "dense", ids=ids, cards=[rows], seed=W, n_valid=nv)
    assert not bool(torch.isin(torch.arange(2900, rows).cuda(), c.uniq).any())
    segs = c.sort(n_valid=torch.tensor([nv], dtype=torch.int32).cuda())
    run_modes(c, segs, f"n_valid W{W}")


@pytest.mark.gpu
@pytest.mark.parametrize("W", REFUSED)
def test_refused_widths_fail_before_any_launch(W):
    ops = _ops()
    c = Case(W, "dense", ids=torch.arange(64).view(-1, 1), cards=[64], seed=1)
    segs = c.sort()
    t = c.table0.clone()
    with pytest.raises(RuntimeError, match="bad width" if W > 2048 else "not a multiple of 4 and > 512"):
        ops.segment_update(segs, ops.RS_UPD_SGD, W, 1, table=t, lr=0.1, dense=c.dense)
    torch.cuda.synchronize()
    _same_bits(t, c.table0, "refused update wrote the table")
    ops.check_status()


# ============================================================================ GPU: one optimizer step per opt.step()
def _step64(w, g, kind, lr, wd, b1=0.9, b2=0.999, eps=1e-8):
    """one float64 step from zero moments on the summed gradient (lazy: touched rows only)"""
    g = g + wd * w
    if kind == "sgd":
        return w - lr * g, None, None
    m, v = (1 - b1) * g, (1 - b2) * g * g
    return w - lr / (1 - b1) * (m / (v.sqrt() / np.sqrt(1 - b2) + eps)), m, v


def _field_models(name, cards):
    from deeplearningrecommendationsystem_b200.nfield import FieldFFM, FieldFM
    cls, D = (FieldFM, 16) if name == "fm" else (FieldFFM, 8)
    return cls(cards, D, fused=True, seed=3, device="cuda"), cls(cards, D, fused=False, seed=3, device="cuda")


def _dropin_models(name):
    from deeplearningrecommendationsystem_b200 import model as M
    torch.manual_seed(3)
    dense = (M.MatrixFactorization(300, 500, 32) if name == "mf" else M.DIN(500, 16)).cuda()
    return copy.deepcopy(dense).fuse_embedding_updates(), dense


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["adam", "sgd"])
@pytest.mark.parametrize("name", ["fm", "ffm", "mf", "din"])
def test_two_forwards_then_one_step(name, kind):
    """two forwards on different batches that share rows, one opt.step(): one step of the optimizer (wd = 1e-2) on the
    summed gradient, as torch.optim takes one step on the accumulated .grad -- the moments advance once, the decay is
    applied once.  The summed gradient comes from the same model in its dense-gradient mode."""
    from deeplearningrecommendationsystem_b200 import ops
    from deeplearningrecommendationsystem_b200.optim import FusedRowOptimizer
    lr, wd, B = 0.05, 1e-2, 256
    g = torch.Generator().manual_seed(9)
    bce = torch.nn.BCELoss()
    if name in ("fm", "ffm"):
        cards = [5, 40, 300, 17]
        fused, dense = _field_models(name, cards)
        batches = [(torch.stack([torch.randint(0, c, (B,), generator=g) for c in cards], dim=1).cuda(),) for _ in range(2)]
        ys = [(torch.rand(B, 1, generator=g) < 0.3).float().cuda() for _ in range(2)]
        offs = torch.tensor(fused.offsets_host).cuda()
        keys = torch.cat([b[0] + offs for b in batches]).reshape(-1)
        tab_f, dense_tabs = (lambda: fused.weight.data), [dense.weight]
    else:
        fused, dense = _dropin_models(name)
        if name == "mf":
            batches = [(torch.randint(0, 300, (B,), generator=g).cuda(), torch.randint(0, 500, (B,), generator=g).cuda()) for _ in range(2)]
            ys = [(torch.rand(B, generator=g) < 0.4).float().cuda() for _ in range(2)]
            keys = torch.cat([torch.cat([u, i + 300]) for u, i in batches])
            tab_f = lambda: torch.cat([fused.user_embeddings.weight.data, fused.item_embeddings.weight.data])    # noqa: E731
            dense_tabs = [dense.user_embeddings.weight, dense.item_embeddings.weight]
        else:
            batches = [(torch.randint(0, 500, (B, 12), generator=g).cuda(), torch.randint(0, 500, (B,), generator=g).cuda())
                       for _ in range(2)]
            ys = [(torch.rand(B, 1, generator=g) < 0.4).float().cuda() for _ in range(2)]
            keys = torch.cat([torch.cat([h.reshape(-1), t]) for h, t in batches])
            tab_f, dense_tabs = (lambda: fused.item_embedding.weight.data), [dense.item_embedding.weight]
    touched = torch.unique(keys)
    assert touched.numel() < keys.numel()                          # the batches share rows
    w0 = tab_f().clone()
    assert torch.equal(w0, torch.cat([t.detach() for t in dense_tabs]))
    opt = FusedRowOptimizer(fused, None, lr=lr, kind=kind, weight_decay=wd)
    opt.zero_grad()
    sum(bce(fused(*b), y) for b, y in zip(batches, ys)).backward()
    opt.step()
    ops.check_status()
    loss = sum(bce(dense(*b), y) for b, y in zip(batches, ys))
    gsum = torch.cat(torch.autograd.grad(loss, dense_tabs))
    w64, m64, v64 = _step64(w0[touched].double(), gsum[touched].double(), kind, lr, wd)
    got = tab_f()
    np.testing.assert_allclose(got[touched].cpu().numpy(), w64.cpu().numpy(), rtol=1e-5, atol=1e-6, err_msg=f"{name} {kind}")
    mask = torch.ones(w0.shape[0], dtype=torch.bool, device="cuda")
    mask[touched] = False
    _same_bits(got[mask], w0[mask], f"{name} {kind}: untouched rows")
    if kind == "adam":
        mm = fused.adam_m if name in ("fm", "ffm") else fused._row_sink.groups[0]["m"]
        np.testing.assert_allclose(mm[touched].cpu().numpy(), m64.cpu().numpy(), rtol=1e-5, atol=1e-9, err_msg=f"{name} m")


@pytest.mark.gpu
def test_two_forwards_without_a_stash_refuse_weight_decay(monkeypatch):
    """the stash-free FFM forward (RS_FFM_RECOMPUTE=1) rebuilds its gradient from the table at the step, so it cannot be
    merged with a second forward; with weight decay that must raise instead of decaying twice"""
    from deeplearningrecommendationsystem_b200.nfield import FieldFFM
    from deeplearningrecommendationsystem_b200.optim import FusedRowOptimizer
    monkeypatch.setenv("RS_FFM_RECOMPUTE", "1")
    cards = [5, 40, 300, 17]
    m = FieldFFM(cards, 8, fused=True, seed=3, device="cuda")
    opt = FusedRowOptimizer(m, None, lr=0.05, weight_decay=1e-2)
    assert m._recompute
    g = torch.Generator().manual_seed(2)
    ids = [torch.stack([torch.randint(0, c, (64,), generator=g) for c in cards], dim=1).cuda() for _ in range(2)]
    (m(ids[0]).sum() + m(ids[1]).sum()).backward()
    with pytest.raises(RuntimeError, match="RS_FFM_RECOMPUTE=0"):
        opt.step()


def _sharded_adam(world, kind, steps=2, forwards=1):
    from deeplearningrecommendationsystem_b200 import dist as rsdist
    from deeplearningrecommendationsystem_b200.nfield import FieldFFM, FieldFM
    from deeplearningrecommendationsystem_b200.optim import FusedRowOptimizer
    cards = [3, 50, 7, 1000, 24, 12, 301, 5]
    cls, D = (FieldFM, 16) if kind == "fm" else (FieldFFM, 8)
    B, lr, wd = 300, 0.01, 1e-2
    ref = cls(cards, D, fused=True, seed=4, device="cpu")
    bce = torch.nn.BCELoss()

    def batch(rank, step):
        g = torch.Generator().manual_seed(700 + 10 * rank + step)
        ids = torch.stack([(torch.rand(B, generator=g) ** 2 * c).long().clamp_(max=c - 1) for c in cards], dim=1)
        return ids.cuda(), (torch.rand(B, 1, generator=g) < 0.3).float().cuda()

    def rank_fn(fab):
        m = cls(cards, D, fused=True, seed=4, device="cuda", sharded=True, fabric=fab, replicate_below=0)
        m.load_global(ref.weight.data)
        opt = FusedRowOptimizer(m, torch.optim.SGD([m.bias], lr=lr), lr=lr, kind="adam", weight_decay=wd)
        for s in range(steps):
            ids, y = batch(fab.rank, s)
            opt.zero_grad()
            sum(bce(m(ids), y) for _ in range(forwards)).backward()
            opt.step()
        return m.weight.data.clone(), m.adam_m.clone(), m.adam_v.clone(), m

    outs = rsdist.ThreadFabric.run(world, rank_fn)
    m = cls(cards, D, fused=True, seed=4, device="cpu").cuda()
    opt = FusedRowOptimizer(m, torch.optim.SGD([m.bias], lr=lr), lr=lr, kind="adam", weight_decay=wd)
    for s in range(steps):
        bs = [batch(r, s) for r in range(world)]
        opt.zero_grad()
        bce(m(torch.cat([b[0] for b in bs])), torch.cat([b[1] for b in bs])).backward()
        opt.step()
    for k, want in ((0, m.weight.data), (1, m.adam_m), (2, m.adam_v)):
        got = outs[0][3].assemble_global([o[k] for o in outs])
        np.testing.assert_allclose(got.cpu().numpy(), want.cpu().numpy(), rtol=1e-5, atol=(2e-6, 1e-9, 1e-12)[k],
                                   err_msg=f"world {world} {kind}: {('w', 'm', 'v')[k]}")


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["fm", "ffm"])
@pytest.mark.parametrize("world", [2, 4])
def test_row_sharded_adam_with_weight_decay_equals_single_gpu(world, kind):
    """every table row-sharded (replicate_below=0) on virtual ranks: the owners run lazy Adam with weight decay over their
    n_valid-padded receive lists; two steps equal the single-GPU steps on the concatenated batch"""
    from deeplearningrecommendationsystem_b200 import ops
    _sharded_adam(world, kind)
    ops.check_status()


@pytest.mark.gpu
def test_row_sharded_two_forwards_with_adam_raise():
    with pytest.raises(RuntimeError, match="one forward per optimizer step"):
        _sharded_adam(2, "fm", steps=1, forwards=2)
