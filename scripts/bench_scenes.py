"""Many scenes per tracker step: a Python loop of PointReidentifier.step (one scene per call) against one
MultiScenePointReidentifier.step over the same seeded scenes, in 'parity_tc' mode with the 'pt' model, 128 points per object.

S in {1, 8, 32, 128} scenes.  Each scene draws its track count T_s and detection count D_s around 32 (uniform in [24, 40]) or
around 128 (uniform in [96, 160]), half the scenes each; its sweep has 30 000 points (tests/test_frontend_oracle.scene).
Sample ranks are explicit and shared by both paths, and their outputs and banks are compared for identity in the same run
("identical").  Every repetition starts from copies of the same banks.

Times: CUDA events around the whole step (median over --reps after --warmup steps), and per phase -- front-end, encode,
score, assign, bank update -- from events recorded around each phase's calls in a separate set of repetitions (the events
add a little host time per call).  Phase times include the host time the GPU waits for launches: at these sizes the step
is launch-bound.  Then linear_assignment_blocks against linear_assignment on the same problems padded to (S, Tmax, Dmax)
(padding masked out).  Writes a header line (GPU name, power limit, read in the same run) and one JSON line per S to --out."""
import argparse
import copy
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import helpers  # noqa: E402
from oracle import reid_oracle as O  # noqa: E402
from test_frontend_oracle import scene  # noqa: E402

import pcreid_b200.kernels as K  # noqa: E402
import pcreid_b200.models.tracking as TR  # noqa: E402

DEV = "cuda"
MIN_SCORE = -2.0
NPTS = 128


def gpu_header():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1], "torch": torch.__version__,
            "mode": "parity_tc", "model": "pt (128, 64, 32)", "points_per_object": NPTS, "min_score": MIN_SCORE}


def make_scenes(model, S, seed):
    rng = np.random.default_rng(seed)
    banks, frames, ranks = [], [], []
    for s in range(S):
        lo, hi = (24, 40) if s % 2 == 0 else (96, 160)
        T, D = int(rng.integers(lo, hi + 1)), int(rng.integers(lo, hi + 1))
        x, h = model.encode(O.synth_objects(T, NPTS, seed * 1000 + s).to(DEV))
        bank = TR.PointFeatureSet()
        bank.store_new(x, h, torch.full((T,), 64, device=DEV))
        pts, boxes = scene(30000, D, seed * 1000 + s)
        dl = torch.from_numpy(rng.integers(0, 8, D)).to(DEV)
        frames.append((torch.from_numpy(pts).to(DEV), torch.from_numpy(boxes).to(DEV), dl, torch.arange(T, device=DEV),
                       torch.from_numpy(rng.integers(0, 8, T)).to(DEV)))
        ranks.append(torch.randint(0, 1 << 30, (D, NPTS), generator=torch.Generator().manual_seed(s)).to(DEV))
        banks.append(bank)
    return banks, frames, ranks


def run_loop(model, banks, frames, ranks):
    return [TR.PointReidentifier(model, b).step(*f, MIN_SCORE, sample_rank=r) for b, f, r in zip(banks, frames, ranks)]


def run_multi(model, banks, frames, ranks):
    return TR.MultiScenePointReidentifier(model, banks).step(frames, MIN_SCORE, sample_ranks=ranks)


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1), out


class PhaseTimer:
    """wraps the calls of each phase with CUDA events (monkeypatched for the duration of a `with` block)"""
    PHASES = {"front_end": [(TR, "crop_center_resample"), (TR, "crop_center_resample_scenes")],
              "assign": [(K, "linear_assignment"), (K, "linear_assignment_blocks")],
              "bank_update": [(TR.PointFeatureSet, "replace_old"), (TR.PointFeatureSet, "store_new")]}

    def __init__(self, model):
        self.targets = dict(self.PHASES, encode=[(model, "encode")], score=[(model, "match_all_pairs"), (model, "match_pairs")])
        self.events, self.saved = [], []

    def _wrap(self, phase, fn):
        def wrapped(*a, **kw):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out = fn(*a, **kw)
            e1.record()
            self.events.append((phase, e0, e1))
            return out
        return wrapped

    def __enter__(self):
        for phase, lst in self.targets.items():
            for obj, name in lst:
                orig = getattr(obj, name)
                self.saved.append((obj, name, orig))
                setattr(obj, name, self._wrap(phase, orig))
        return self

    def __exit__(self, *exc):
        for obj, name, orig in reversed(self.saved):
            if isinstance(obj, torch.nn.Module):
                delattr(obj, name)            # the model's own methods again
            else:
                setattr(obj, name, orig)      # module function / class function
        self.saved = []

    def totals(self):
        torch.cuda.synchronize()
        out = {p: 0.0 for p in self.targets}
        for phase, e0, e1 in self.events:
            out[phase] += e0.elapsed_time(e1)
        self.events = []
        return out


def identical(a_res, b_res, a_banks, b_banks):
    for ra, rb, ba, bb in zip(a_res, b_res, a_banks, b_banks):
        for x, y in zip(ra, rb):
            if (x is None) != (y is None) or (x is not None and not torch.equal(x, y)):
                return False
        if not (torch.equal(ba.pts_feats, bb.pts_feats) and torch.equal(ba.pts_xyz, bb.pts_xyz)
                and torch.equal(ba.lengths, bb.lengths)):
            return False
    return True


def bench_blocks(costs, frames, reps):
    """linear_assignment_blocks against padded (S, Tmax, Dmax) linear_assignment on the step's own cost matrices, gated by
    class only"""
    shapes = [tuple(c.shape) for c in costs]
    Tm, Dm = max(t for t, _ in shapes), max(d for _, d in shapes)
    score = torch.cat([c.reshape(-1) for c in costs])
    gates = [TR.class_gate(f[2], f[4], None, None, use_lengths=False) for f in frames]
    gate = torch.cat([g.reshape(-1) for g in gates])
    pad = torch.zeros((len(costs), Tm, Dm), device=DEV)
    pmask = torch.zeros((len(costs), Tm, Dm), device=DEV, dtype=torch.bool)
    for b, (c, g) in enumerate(zip(costs, gates)):
        pad[b, :c.shape[0], :c.shape[1]] = c
        pmask[b, :c.shape[0], :c.shape[1]] = g
    blk = lambda: K.linear_assignment_blocks(score, shapes, MIN_SCORE, gate)
    padded = lambda: K.linear_assignment(pad, MIN_SCORE, pmask)
    for _ in range(2):
        blk(), padded()
    tb, tp = [], []
    for _ in range(reps):
        tb.append(timed(blk)[0])
        tp.append(timed(padded)[0])
    _, (_, t4d) = timed(blk)
    _, (_, t4d_p) = timed(padded)
    c0, same = 0, True
    for b, (t, d) in enumerate(shapes):
        same &= torch.equal(t4d[c0:c0 + d], t4d_p[b, :d])
        c0 += d
    return {"blocks_ms": statistics.median(tb), "padded_ms": statistics.median(tp), "padded_shape": [len(costs), Tm, Dm],
            "pairs_packed": score.numel(), "pairs_padded": pad.numel(), "padded_result_equal": bool(same)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scenes", default="1,8,32,128")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    model, _ = helpers.build_pair("pt", (128, 64, 32), device=DEV)
    model.set_mode("parity_tc")
    lines = [gpu_header()]
    print(json.dumps(lines[0]), flush=True)
    for S in [int(x) for x in a.scenes.split(",")]:
        banks, frames, ranks = make_scenes(model, S, seed=S)
        loop_b, multi_b = copy.deepcopy(banks), copy.deepcopy(banks)
        ref = run_loop(model, loop_b, frames, ranks)
        got = run_multi(model, multi_b, frames, ranks)
        same = identical(got, ref, multi_b, loop_b)
        for _ in range(a.warmup):
            run_loop(model, copy.deepcopy(banks), frames, ranks)
            run_multi(model, copy.deepcopy(banks), frames, ranks)
        t_loop, t_multi = [], []
        for _ in range(a.reps):                                    # alternated
            b = copy.deepcopy(banks)
            t_loop.append(timed(lambda: run_loop(model, b, frames, ranks))[0])
            b = copy.deepcopy(banks)
            t_multi.append(timed(lambda: run_multi(model, b, frames, ranks))[0])
        phases = {}
        for name, fn in (("loop", run_loop), ("multi", run_multi)):
            per = []
            for _ in range(a.reps):
                b = copy.deepcopy(banks)
                with PhaseTimer(model) as pt:
                    timed(lambda: fn(model, b, frames, ranks))
                per.append(pt.totals())
            phases[name] = {k: round(statistics.median(p[k] for p in per), 3) for k in per[0]}
        row = {"S": S, "tracks": sum(len(f[3]) for f in frames), "detections": sum(f[1].shape[0] for f in frames),
               "identical": bool(same), "loop_ms": round(statistics.median(t_loop), 3),
               "multi_ms": round(statistics.median(t_multi), 3),
               "speedup": round(statistics.median(t_loop) / statistics.median(t_multi), 3),
               "loop_ms_all": [round(t, 3) for t in t_loop], "multi_ms_all": [round(t, 3) for t in t_multi],
               "phases_ms": phases, "assign": bench_blocks([r[2] for r in ref], frames, a.reps)}
        lines.append(row)
        print(json.dumps(row), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            for ln in lines:
                f.write(json.dumps(ln) + "\n")


if __name__ == "__main__":
    main()
