"""Tracks kept on the device: MultiScenePointReidentifier.step (one PointFeatureSet per scene, every bank row an active
track, the caller rebuilding track_index / track_labels on the host) against ReIDTracker.step (TrackTable, max_age=None), over
the same seeded sequence of frames, in 'parity_tc' mode with the 'pt' model, 128 points per object.

S in {1, 8, 32, 128} scenes with the scenes of bench_scenes.make_scenes (D_s uniform in [24, 40] or [96, 160], 30 000-point
sweeps).  Every frame re-detects the same boxes of the same sweep with fresh sample ranks, so most detections find their track
and the banks stay near D_s rows; the scenes start without tracks.  Both classes' outputs are compared frame by frame
("identical": same track ids -- a bank row is a slot when nothing retires -- and same costs).

Times: CUDA events around each step, the median over the frames after the first --warmup, the two classes alternated frame by
frame.  Phases in a second pass of the sequence (events around each phase's calls; they include the host time the GPU waits
for launches): front_end, encode, score, assign, and for the bank / table work
  gate:        class_gate (per scene)                          | kernels.track_gate_blocks
  bank_update: PointFeatureSet.replace_old + store_new          | kernels.track_update + kernels.track_scatter
and "outside" = step total - the sum of the phases.  Then the sequence once more with max_age=2 and a capacity of
twice the largest D_s for the tracker (the banks of MultiScenePointReidentifier only grow): bank bytes after the last frame.  Writes a header line (GPU name, power limit and
clocks read in the same run) and one JSON line per S to --out.

--motion: instead, ReIDTracker with MotionModel() (AB3DMOT's defaults, dt = 1) against ReIDTracker without a motion model over
the same sequence, alternated frame by frame, ids and alive tracks per frame compared; the phase pass adds "predict"
(kernels.track_predict) and "correct" (kernels.track_correct), and "gate" covers kernels.track_gate_motion_blocks.  The boxes
do not move, but the two trackers need not agree: without a bound a detection may match any track of its class, while the
Mahalanobis bound leaves it only the tracks near its box, so a detection whose own track scores <= min_score starts a new
track, and the step then scores more tracks."""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import torch  # noqa: E402

from bench_scenes import DEV, MIN_SCORE, NPTS, PhaseTimer, gpu_header, make_scenes  # noqa: E402  (also puts tests/ on the path)
import helpers  # noqa: E402

import pcreid_b200.kernels as K  # noqa: E402
import pcreid_b200.models.tracking as TR  # noqa: E402


class TablePhaseTimer(PhaseTimer):
    PHASES = dict(PhaseTimer.PHASES, gate=[(TR, "class_gate"), (K, "track_gate_blocks")],
                  bank_update=[(TR.PointFeatureSet, "replace_old"), (TR.PointFeatureSet, "store_new"), (K, "track_update"),
                               (K, "track_scatter")])


class MotionPhaseTimer(TablePhaseTimer):
    PHASES = dict(TablePhaseTimer.PHASES, gate=TablePhaseTimer.PHASES["gate"] + [(K, "track_gate_motion_blocks")],
                  predict=[(K, "track_predict")], correct=[(K, "track_correct")])


def sequence(model, S, frames):
    """the scenes of make_scenes, re-detected every frame with fresh ranks -> [[(sweep, boxes, labels)] per frame], ranks"""
    _, base, _ = make_scenes(model, S, seed=S)
    g = torch.Generator().manual_seed(S)
    dets = [[(f[0], f[1], f[2]) for f in base] for _ in range(frames)]
    ranks = [[torch.randint(0, 1 << 30, (f[1].shape[0], NPTS), generator=g).to(DEV) for f in base] for _ in range(frames)]
    return dets, ranks


class Multi:
    """MultiScenePointReidentifier with every bank row active, track_index / track_labels kept by the caller"""

    def __init__(self, model, S):
        self.banks = [TR.PointFeatureSet() for _ in range(S)]
        self.labels = [torch.zeros(0, dtype=torch.int64, device=DEV) for _ in range(S)]
        self.reid = TR.MultiScenePointReidentifier(model, self.banks)

    def step(self, dets, ranks):
        frames = [(w, b, l, torch.arange(len(bank), device=DEV), lab) for (w, b, l), bank, lab in zip(dets, self.banks, self.labels)]
        out = self.reid.step(frames, MIN_SCORE, sample_ranks=ranks)
        for s, (tfd, new_rows, _) in enumerate(out):
            self.labels[s] = torch.cat([self.labels[s], dets[s][2][tfd < 0]])
        return out

    def nbytes(self):
        return sum(t.numel() * t.element_size() for b in self.banks for t in (b.pts_xyz, b.pts_feats, b.lengths) if t is not None)


def table_bytes(table):
    names = [n for n, _, _ in K.TRACK_SLOT_FIELDS] + [n for n, _ in K.TRACK_SCENE_FIELDS] + ["xyz", "feat"]
    return sum(getattr(table, n).numel() * getattr(table, n).element_size() for n in names)


def same(multi_out, tracker_out):
    for (tfd, new_rows, cost), (ids, c) in zip(multi_out, tracker_out):
        want = tfd.clone()
        want[tfd < 0] = new_rows
        if not torch.equal(want, ids) or (cost is None) != (c is None) or (cost is not None and not torch.equal(cost, c)):
            return False
    return True


def timed_step(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1), out


def motion_rows(model, a):
    """--motion: one JSON line per S, the tracker with MotionModel() against the tracker without one"""
    for S in [int(x) for x in a.scenes.split(",")]:
        dets, ranks = sequence(model, S, a.frames)
        capacity = min(K.TRACK_MAX_CAPACITY, a.frames * max(d[1].shape[0] for d in dets[0]))
        make = {"plain": lambda: TR.ReIDTracker(model, num_scenes=S, capacity=capacity),
                "motion": lambda: TR.ReIDTracker(model, num_scenes=S, capacity=capacity, motion=TR.MotionModel())}
        # timed pass, alternated frame by frame; ids compared
        trackers = {k: f() for k, f in make.items()}
        times, identical, alive = {k: [] for k in make}, True, {k: [] for k in make}
        for f in range(a.frames):
            out = {}
            for k, tr in trackers.items():
                t, out[k] = timed_step(lambda: tr.step(dets[f], MIN_SCORE, sample_ranks=ranks[f], dt=1.0))
                alive[k].append(int(tr.table.count.sum()))
                if f >= a.warmup:
                    times[k].append(t)
            identical &= all(torch.equal(x[0], y[0]) for x, y in zip(out["plain"], out["motion"]))
        # phase pass
        phases = {}
        for k, f_make in make.items():
            tr, per = f_make(), []
            for f in range(a.frames):
                with MotionPhaseTimer(model) as pt:
                    total, _ = timed_step(lambda: tr.step(dets[f], MIN_SCORE, sample_ranks=ranks[f], dt=1.0))
                p = pt.totals()
                p["outside"] = total - sum(p.values())
                p["step"] = total
                if f >= a.warmup:
                    per.append(p)
            phases[k] = {n: round(statistics.median(p[n] for p in per), 3) for n in per[0]}
        del trackers, tr
        med = {k: statistics.median(v) for k, v in times.items()}
        yield {"S": S, "detections_per_frame": sum(d[1].shape[0] for d in dets[0]), "capacity": capacity,
               "identical_ids": bool(identical), "alive_tracks_per_frame": alive, "plain_ms": round(med["plain"], 3), "motion_ms": round(med["motion"], 3),
               "motion_minus_plain_ms": round(med["motion"] - med["plain"], 3),
               "plain_ms_all": [round(t, 3) for t in times["plain"]], "motion_ms_all": [round(t, 3) for t in times["motion"]],
               "phases_ms": phases}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scenes", default="1,8,32,128")
    ap.add_argument("--frames", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--motion", action="store_true", help="the tracker with a motion model against the tracker without")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    model, _ = helpers.build_pair("pt", (128, 64, 32), device=DEV)
    model.set_mode("parity_tc")
    lines = [dict(gpu_header(), frames=a.frames)]
    print(json.dumps(lines[0]), flush=True)
    for row in (motion_rows(model, a) if a.motion else ()):
        lines.append(row)
        print(json.dumps(row), flush=True)
    for S in ([] if a.motion else [int(x) for x in a.scenes.split(",")]):
        dets, ranks = sequence(model, S, a.frames)
        capacity = min(K.TRACK_MAX_CAPACITY, a.frames * max(d[1].shape[0] for d in dets[0]))
        # timed pass, alternated frame by frame; outputs compared
        multi, tracker = Multi(model, S), TR.ReIDTracker(model, num_scenes=S, capacity=capacity)
        t_multi, t_table, identical, tracks = [], [], True, []
        for f in range(a.frames):
            tm, out_m = timed_step(lambda: multi.step(dets[f], ranks[f]))
            tt, out_t = timed_step(lambda: tracker.step(dets[f], MIN_SCORE, sample_ranks=ranks[f]))
            identical &= same(out_m, out_t)
            if f >= a.warmup:
                t_multi.append(tm)
                t_table.append(tt)
            tracks.append(sum(len(b) for b in multi.banks))
        # phase pass
        phases = {}
        for name in ("multi", "table"):
            obj = Multi(model, S) if name == "multi" else TR.ReIDTracker(model, num_scenes=S, capacity=capacity)
            per = []
            for f in range(a.frames):
                with TablePhaseTimer(model) as pt:
                    total, _ = timed_step(lambda: obj.step(dets[f], ranks[f]) if name == "multi"
                                          else obj.step(dets[f], MIN_SCORE, sample_ranks=ranks[f]))
                p = pt.totals()
                p["outside"] = total - sum(p.values())
                p["step"] = total
                if f >= a.warmup:
                    per.append(p)
            phases[name] = {k: round(statistics.median(p[k] for p in per), 3) for k in per[0]}
        # retirement: the tracker with max_age=2 against the growing banks
        capacity2 = min(K.TRACK_MAX_CAPACITY, 2 * max(d[1].shape[0] for d in dets[0]))
        multi2, tracker2 = Multi(model, S), TR.ReIDTracker(model, num_scenes=S, capacity=capacity2, max_age=2)
        for f in range(a.frames):
            multi2.step(dets[f], ranks[f])
            tracker2.step(dets[f], MIN_SCORE, sample_ranks=ranks[f])
        torch.cuda.synchronize()
        retired = {"capacity": capacity2, "multi_bank_bytes": multi2.nbytes(), "table_bytes": table_bytes(tracker2.table),
                   "table_alive": int(tracker2.table.count.sum()), "multi_rows": sum(len(b) for b in multi2.banks),
                   "table_dropped": int(tracker2.table.dropped.sum())}
        del multi, tracker, obj, multi2, tracker2
        row = {"S": S, "detections_per_frame": sum(d[1].shape[0] for d in dets[0]), "capacity": capacity,
               "bank_rows_per_frame": tracks, "identical": bool(identical),
               "multi_ms": round(statistics.median(t_multi), 3), "table_ms": round(statistics.median(t_table), 3),
               "speedup": round(statistics.median(t_multi) / statistics.median(t_table), 3),
               "multi_ms_all": [round(t, 3) for t in t_multi], "table_ms_all": [round(t, 3) for t in t_table],
               "phases_ms": phases,
               "max_age_2": retired}
        lines.append(row)
        print(json.dumps(row), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            for ln in lines:
                f.write(json.dumps(ln) + "\n")


if __name__ == "__main__":
    main()
