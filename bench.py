#!/usr/bin/env python
"""bench.py -- headline benchmark of the hot path (BASELINE.json: "pair scores/sec + objects encoded/sec
(PT, 256 pts)"), configs[1]: Point Transformer (pts_point-transformer_r_nus_det) inference, 1024 tracks +
1024 detections x 256 points, 1024 x 1024 all-pairs `xcorr_eff` match per GPU.

A step = encode the step's tracks and detections (PT backbone) + score every track x detection pair.
At N GPUs the track rows are sharded (weak scaling: 1024 tracks per rank, the 1024 detections are
split for encoding and all-gathered once).  Prints ONE JSON line (rank 0).

The headline mode is 'parity_tc' -- every contraction on the tensor cores at an 11-bit significand (tf32 encoder GEMMs,
fp16 matcher operands), the mode that passes the parity gates of SURVEY.md 8d; the line carries the measured parity
(`parity`: max |dlogit| and RAW top-1 agreement on a 256 x 256 block of the workload against the CPU oracle), the bf16
'fast' mode beside it (`fast_mode`), an encoder roofline (`encoder`), and a fixed-size strong-scaling leg (`strong`: 4096 x 4096
pairs row-sharded over the N ranks INCLUDING the all-gather of the score rows).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--mode parity_tc|fast|parity] [--dump-outputs DIR]

--dump-outputs DIR writes the score rows the timed path returned in its last step, one file per rank, so that two builds can
be compared output for output on identical seeded inputs.
"""
import argparse
import glob
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

T_PER_GPU, D_TOTAL, NPTS = 1024, 1024, 256
BLIST = (256, 128, 64)
STRONG_T = STRONG_D = 4096
# algorithmic work of the reference formulation (BASELINE.md section 3, torch.utils.flop_counter on the reference)
FLOP_PER_OBJECT = 592e6          # Pointnet_Backbone @256 pts
FLOP_PER_PAIR = 101.25e6         # xcorr_eff + pool + head @256 pts
# The bench line is BASELINE.json configs[1] ("c2", the configuration the metric is quoted on).  --config runs the other
# named single-box configurations through the same protocol (they are parity-test cases, not the headline):
#   c3 = configs[2]: DGCNN (k = 20), 2048 + 2048 objects x 256 pts, 2048 x 2048 matrix, FIXED size sharded over the ranks
#   c4 = configs[3]: Point Transformer, 4096 + 4096 objects x 1024 pts, 4096 x 4096 matrix, FIXED size sharded over the ranks
CONFIGS = {
    "c2": dict(kind="pt", npts=256, tracks=1024, dets=1024, scaling="weak", flop_obj=592e6, flop_pair=101.25e6, tag="configs[1]: Point Transformer"),
    "c3": dict(kind="dgcnn", npts=256, tracks=2048, dets=2048, scaling="strong", flop_obj=1.98e9, flop_pair=101.25e6, tag="configs[2]: DGCNN k=20"),
    "c4": dict(kind="pt", npts=1024, tracks=4096, dets=4096, scaling="strong", flop_obj=4 * 592e6, flop_pair=4 * 101.25e6,
               tag="configs[3]: Point Transformer (Waymo dense shape)"),
}
METRIC = "pair scores/sec (PT-256 encode + all-pairs xcorr_eff match)"
CPU_SAMPLE = (64, 8192)          # objects per side, pairs: the bounded CPU sample, identical in both arms
MODE_TEXT = {
    "parity_tc": "parity_tc: tensor cores at an 11-bit significand -- tcgen05 kind::tf32 SA shared MLPs / Self_Attention blocks in the "
                 "encoder with operands pre-rounded to tf32 (the three FP_SA blocks that emit the embedding stay fp32: they cost ~1 % "
                 "raw top-1, profiles/r02_parity_error_budget.md), fused kind::f16 matcher with fp16 operands (pair_tc.cu, pair_tc2.cu) "
                 "-- fp32 accumulate / norms; gate |dlogit| <= 5e-3, raw top-1 >= 0.97",
    "fast": "fast: the same kernels with bf16 matcher operands; gate |dlogit| <= 3e-2",
    "parity": "parity: fp32 FFMA kernels, logits within 1e-4 of the reference",
    "parity_x3": "parity_x3: the parity path with its Linears / 1x1 convs on tcgen05 at fp32-grade accuracy (TMA-staged 3 x tf32 GEMM, "
                 "cn_linear_tma.cu), logits within 1e-4 of the reference",
}
DTYPE = {"parity_tc": "f16", "fast": "bf16", "parity": "f32", "parity_x3": "tf32x3"}
DUMP_BYTES = 64 * 10**6          # --dump-outputs: at most this many bytes over all files of all ranks


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d, "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


def ncu_traffic(mode):
    """per-unit DRAM bytes of the fused kernels from the newest ncu --set full capture (profiles/rNN_ncu_traffic.json, written by
    scripts/ncu_traffic.py from the capture itself) -> ({kernel: bytes per (pair, direction) unit}, source) or (None, None)."""
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_ncu_traffic.json")))
    if not files:
        return None, None
    d = json.load(open(files[-1]))
    ent = d.get("modes", {}).get(mode) or d.get("modes", {}).get("parity_tc") or d.get("modes", {}).get("fast")
    if not ent:
        return None, None
    return {k: v["dram_bytes_per_unit"] for k, v in ent["kernels"].items()}, os.path.relpath(files[-1], ROOT)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm = sorted(int(float(r[1])) for r in self.rows if len(r) >= 8 and r[1].replace('.', '').isdigit())
        mx = [int(float(r[2])) for r in self.rows if len(r) >= 8 and r[2].replace('.', '').isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 8 for n, v in zip(names, r[4:8]) if v.lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx[0] if mx else None, "reasons": reasons,
                "samples": len(sm)}


_ORACLE = {}


def _oracle():
    """the CPU checker: oracle restatement of the reference's PyTorch path (bit-exact vs the reference modules,
    tests/test_reidnet_pinned.py) with the weights of the benchmarked model (seed 66, default init)."""
    if "orc" not in _ORACLE:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import helpers                                  # oracle builder shared with the parity tests
        from oracle import reid_oracle as O
        _ORACLE["orc"] = helpers.build_pair("pt", BLIST, device="cpu", perturb=False)[1]
        _ORACLE["O"] = O
    return _ORACLE["orc"], _ORACLE["O"]


def cpu_reference_sample(n_obj=CPU_SAMPLE[0], n_pairs=CPU_SAMPLE[1], threads=None, warm=True):
    """The reference's PyTorch path (oracle port) on host cores, on a bounded sample of the same workload: encode
    n_obj+n_obj objects, score n_pairs pairs; extrapolated to the step's composition (objects and pairs per step).
    warm: one small untimed pass first (thread pool, allocator, lazy module state), so a single call is not a cold number."""
    orc, O = _oracle()
    threads = threads or os.cpu_count()
    torch.set_num_threads(threads)
    if warm:
        w = O.synth_objects(4, NPTS, 7)
        xw, hw = orc.encode(w)
        orc.match_all_pairs(hw, xw, hw, xw, chunk=4096)
    t, d = O.synth_objects(n_obj, NPTS, 0), O.synth_objects(n_obj, NPTS, 1)
    t0 = time.perf_counter()
    xt, ht = orc.encode(t)
    xd, hd = orc.encode(d)
    t1 = time.perf_counter()
    rows = max(1, n_pairs // n_obj)
    orc.match_all_pairs(ht[:rows], xt[:rows], hd, xd, chunk=4096)
    t2 = time.perf_counter()
    s_obj = (t1 - t0) / (2 * n_obj)
    s_pair = (t2 - t1) / (rows * n_obj)
    step_s = s_obj * (T_PER_GPU + D_TOTAL) + s_pair * T_PER_GPU * D_TOTAL
    return {"value": T_PER_GPU * D_TOTAL / step_s, "unit": "pairs/s", "cores": threads, "kind": "port",
            "sample": f"{2 * n_obj} objects encoded ({1 / s_obj:.1f} obj/s) + {rows * n_obj} pairs scored ({1 / s_pair:.1f} pairs/s) "
                      f"after one warm-up pass, extrapolated to {T_PER_GPU + D_TOTAL} objects + {T_PER_GPU * D_TOTAL} pairs per step",
            "objects_per_s": 1 / s_obj, "pairs_only_per_s": 1 / s_pair}


def parity_block(model, dev, rows=384, cols=256):
    """measured parity of the benchmarked mode: a rows x cols block of the workload (tracks seed 1000, detections seed 1 --
    the step's own inputs) through the CUDA path end to end (encode + match) against the CPU oracle."""
    orc, O = _oracle()
    from pcreid_b200 import synthetic as S
    t, d = S.synth_objects(rows, NPTS, 1000), S.synth_objects(cols, NPTS, 1)
    torch.set_num_threads(os.cpu_count())
    t0 = time.perf_counter()
    oxt, oht = orc.encode(t)
    oxd, ohd = orc.encode(d)
    Lo = orc.match_all_pairs(oht, oxt, ohd, oxd, chunk=4096)
    cpu_s = time.perf_counter() - t0
    xt, ht = model.encode(t.to(dev))
    xd, hd = model.encode(d.to(dev))
    L = model.match_all_pairs(ht, xt, hd, xd).cpu()
    err = (L - Lo).abs()
    top2 = torch.topk(Lo, 2, dim=1)[0]
    gap = top2[:, 0] - top2[:, 1]
    same = Lo.argmax(1) == L.argmax(1)
    mx = float(err.max())
    dec = gap > 2 * mx
    return {"mode": model.match_mode, "block": f"{rows}x{cols} pairs of the step's own inputs, encode + match end to end vs the CPU oracle",
            "max_abs": mx, "mean_abs": float(err.mean()), "top1_raw": float(same.float().mean()), "decisive_rows": int(dec.sum()),
            "decisive_rows_unchanged": bool(same[dec].all()), "oracle_logit_std": float(Lo.std()), "oracle_gap_median": float(gap.median()),
            "embedding_max_abs": float((ht.cpu() - oht).abs().max()), "oracle_cpu_s": cpu_s}


def dump_scores(out_dir, rows, rank, world):
    """this rank's (T_r, D) score rows as out_dir/scores_rank<r>.npy (float32).  When they exceed the rank's share of DUMP_BYTES,
    a fixed, seeded sample of rows is written instead, with the sampled row indices in scores_rank<r>_rows.npy (float64)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    s = rows.float().cpu()
    path = os.path.join(out_dir, f"scores_rank{rank}")
    keep = (DUMP_BYTES // world - 2 * 128) // (4 * s.shape[1] + 8)          # 128: an .npy header
    if s.shape[0] > keep:
        idx = torch.randperm(s.shape[0], generator=torch.Generator().manual_seed(0))[:keep].sort().values
        s = s[idx]
        np.save(path + "_rows.npy", idx.double().numpy())
    np.save(path + ".npy", s.numpy())


def bench_model(cfg, mode, dev):
    """the benchmarked model: configuration `cfg` (a CONFIGS entry) with its default init under seed 66, in `mode`"""
    from pcreid_b200 import synthetic as S
    n = cfg["npts"]
    torch.manual_seed(66)
    from pcreid_b200.models import build_model
    model = build_model({"pt": S.point_transformer_cfg, "dgcnn": S.dgcnn_cfg}[cfg["kind"]]((n, n // 2, n // 4))).eval().to(dev)
    model.set_mode(mode)
    return model


def bench_inputs(npts, tracks, dets, rank=0, world=1, strong=False):
    """this rank's host (tracks, detections), seeded synthetic objects: its share of `tracks` rows (strong scaling, seed 1000) or
    `tracks` rows of its own (weak scaling, seed 1000 + rank), and its share of the `dets` detections (seed 1)"""
    from pcreid_b200 import synthetic as S
    from pcreid_b200.parallel import shard_range
    if strong:
        t0, t1 = shard_range(tracks, rank, world)
        t = S.synth_objects(tracks, npts, 1000)[t0:t1].contiguous()
    else:
        t = S.synth_objects(tracks, npts, 1000 + rank)
    d0, d1 = shard_range(dets, rank, world)
    return t, S.synth_objects(dets, npts, 1)[d0:d1].contiguous()


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    vals = []
    last = None
    for i in range(args.warmup + args.steps):
        last = cpu_reference_sample(warm=(i == 0))
        if i >= args.warmup:
            vals.append(last["value"])
    v = sum(vals) / len(vals)
    last["value"] = v
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "pairs/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * T_PER_GPU * D_TOTAL / v, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"PT encode {T_PER_GPU}+{D_TOTAL} objects x {NPTS} pts + {T_PER_GPU}x{D_TOTAL} xcorr_eff pairs "
                                   "(reference PyTorch path on host cores, bounded sample per step, extrapolated)"},
            "cpu_baseline": last, "e2e": {"value": v, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--mode", default="parity_tc", choices=["parity", "parity_x3", "parity_tc", "fast"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS), help="which named BASELINE.json configuration (default: the headline c2)")
    ap.add_argument("--tracks", type=int, default=None, help="tracks per GPU (weak configs) / in total (strong configs)")
    ap.add_argument("--dets", type=int, default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the CPU legs (cpu_baseline, parity)")
    ap.add_argument("--no-extra", action="store_true", help="skip the fast-mode and strong-scaling legs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the score rows of the last timed step to DIR/scores_rank<r>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs writes the CUDA path's scores: it needs --impl ours")
    if args.impl == "reference":
        return run_reference(args)

    import torch.distributed as dist
    from pcreid_b200 import _lib, synthetic as S   # the measured legs never import oracle/ or tests/ (CPU checker legs only)
    from pcreid_b200.parallel import encode_and_gather, gathered_bytes, match_all_pairs_sharded, shard_range

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    cfg = CONFIGS[args.config]
    global NPTS, BLIST, FLOP_PER_OBJECT, FLOP_PER_PAIR
    NPTS, BLIST = cfg["npts"], (cfg["npts"], cfg["npts"] // 2, cfg["npts"] // 4)
    FLOP_PER_OBJECT, FLOP_PER_PAIR = cfg["flop_obj"], cfg["flop_pair"]
    strong_main = cfg["scaling"] == "strong"
    T_arg, D = args.tracks or cfg["tracks"], args.dets or cfg["dets"]
    if strong_main:            # fixed matrix: this rank's share of the track rows
        t0_, t1_ = shard_range(T_arg, rank, world)
        T_loc, T_total = t1_ - t0_, T_arg
    else:                      # weak: T_arg track rows on every rank
        T_loc, T_total = T_arg, T_arg * world
    if args.config != "c2":
        args.no_extra = True   # the fast-mode / 4096^2 strong legs belong to the headline configuration
    d0, d1 = shard_range(D, rank, world)
    det_counts = [shard_range(D, r, world)[1] - shard_range(D, r, world)[0] for r in range(world)]

    model = bench_model(cfg, args.mode, dev)
    tracks_h, dets_h = (x.pin_memory() for x in bench_inputs(NPTS, T_arg, D, rank, world, strong_main))
    tracks_d, dets_d = tracks_h.to(dev), dets_h.to(dev)
    out_h = torch.empty((T_loc, D), dtype=torch.float32).pin_memory()

    def step_device():
        return match_all_pairs_sharded(model, tracks_d, dets_d, det_counts)

    def step_e2e():
        t = tracks_h.to(dev, non_blocking=True)
        d = dets_h.to(dev, non_blocking=True)
        rows = match_all_pairs_sharded(model, t, d, det_counts)
        out_h.copy_(rows, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        """-> (total ms, per-step ms, what fn returned in the last step)"""
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
        barrier()
        ev[0].record()
        for i in range(steps):
            out = fn()
            ev[i + 1].record()
        barrier()
        ms = ev[0].elapsed_time(ev[steps])
        t = torch.tensor([ms], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), [ev[i].elapsed_time(ev[i + 1]) for i in range(steps)], out

    for _ in range(args.warmup):
        step_device()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    calls0 = _lib.ABI_CALLS
    total_ms, per_step, rows = timed(step_device, args.steps)
    launches = _lib.ABI_CALLS - calls0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:
        dump_scores(args.dump_outputs, rows, rank, world)
    del rows
    # phase split (device events, extra steps): encode vs match.  Inside the timed steps the ~90 launches of an encoder pass are
    # issued while the previous step's match still runs; measured alone after a synchronize they would be bound by the host's
    # launch rate, so the encode phase is timed as the public API's CUDA-graph replay (ReIDNet.enable_cuda_graphs): device time.
    e0, e1, e2, e3 = (torch.cuda.Event(enable_timing=True) for _ in range(4))
    xt, ht, xd, hd = encode_and_gather(model, tracks_d, dets_d, det_counts)
    torch.cuda.synchronize()
    e0.record()
    model.match_all_pairs(ht, xt, hd, xd)
    e1.record()
    torch.cuda.synchronize()
    match_ms = e0.elapsed_time(e1)
    # per-launch durations of the fused kernels (CUDA events on the launching stream), one more match pass
    kern = {}
    if args.mode in model.TC_MODES:
        fm = model.fused_matcher()
        fm.timing = []
        model.match_all_pairs(ht, xt, hd, xd)
        torch.cuda.synchronize()
        for name, a0, a1, units in fm.timing:
            k = kern.setdefault(name, {"launches": 0, "ms": 0.0, "units": 0})
            k["launches"] += 1
            k["ms"] += a0.elapsed_time(a1)
            k["units"] += units
        fm.timing = None
    del xt, ht, xd, hd
    for _ in range(1):
        step_e2e()
    e2e_ms, _, _ = timed(step_e2e, args.steps)
    # encode phase (after every headline number has been taken: the capture owns a private memory pool)
    model.enable_cuda_graphs(True)
    encode_and_gather(model, tracks_d, dets_d, det_counts)          # capture
    torch.cuda.synchronize()
    e2.record()
    encode_and_gather(model, tracks_d, dets_d, det_counts)
    e3.record()
    torch.cuda.synchronize()
    model.enable_cuda_graphs(False)
    enc_ms = e2.elapsed_time(e3)

    # ---- beside the headline: the bf16 'fast' mode on the same workload (same timing protocol, fewer steps)
    fast = None
    if not args.no_extra and args.mode != "fast":
        model.set_mode("fast")
        for _ in range(2):
            step_device()
        f_ms, _, _ = timed(step_device, min(args.steps, 5))
        fast = {"value": T_total * D / (f_ms / min(args.steps, 5) * 1e-3), "unit": "pairs/s", "ms_per_step": f_ms / min(args.steps, 5),
                "dtype": "bf16", "mode": MODE_TEXT["fast"]}
        model.set_mode(args.mode)

    # ---- strong scaling: a FIXED 4096 x 4096 @256 matrix row-sharded over the ranks, score rows all-gathered inside the timed region
    strong = None
    if not args.no_extra:
        Ts, Ds = STRONG_T, STRONG_D
        s_t0, s_t1 = shard_range(Ts, rank, world)
        s_d0, s_d1 = shard_range(Ds, rank, world)
        s_tc = [shard_range(Ts, r, world)[1] - shard_range(Ts, r, world)[0] for r in range(world)]
        s_dc = [shard_range(Ds, r, world)[1] - shard_range(Ds, r, world)[0] for r in range(world)]
        s_tr = S.synth_objects(Ts, NPTS, 0)[s_t0:s_t1].contiguous().to(dev)
        s_de = S.synth_objects(Ds, NPTS, 1)[s_d0:s_d1].contiguous().to(dev)

        def step_strong():
            return match_all_pairs_sharded(model, s_tr, s_de, s_dc, gather_scores=True, track_counts=s_tc)

        step_strong()
        n_s = 2
        s_ms, _, _ = timed(step_strong, n_s)
        gb = gathered_bytes(model, NPTS, s_dc, s_tc, gather_scores=True)
        strong = {"workload": f"fixed {Ts}x{Ds} all-pairs xcorr_eff @ {NPTS} pts + encode of {Ts}+{Ds} objects, track rows and detections "
                              f"sharded over {world} rank(s); timed region includes the all-gather of the detection embeddings (overlapped "
                              "with scoring of the local detection block) AND the all-gather of the score rows",
                  "scaling": "strong", "steps": n_s, "ms_per_step": s_ms / n_s, "value": Ts * Ds / (s_ms / n_s * 1e-3), "unit": "pairs/s",
                  "bytes_received_per_rank": gb, "mode": args.mode}
        del s_tr, s_de

    if rank == 0:
        pk, pk_src = peaks()
        pairs_total = T_total * D
        ms_step = total_ms / args.steps
        value = pairs_total / (ms_step * 1e-3)
        n_enc = T_loc + (d1 - d0)
        match_tflops = FLOP_PER_PAIR * T_loc * D / (match_ms * 1e-3) / 1e12 if match_ms > 0 else None
        peak_tf = pk["bf16_tflops_sustained"]
        roof_kernel = "match stage (cn_linear_kernel<*> dominates; unfused fp32 parity path)"
        roof_extra, roof_traffic, traffic_src = {}, None, None
        if kern:
            # dominant kernels: the three fused phases; algorithmic FLOPs of the reference formulation (101.25 MFLOP/pair:
            # stage 1 both ways = 33.9 %, stage 2 + pool + head = 66.1 %) / their summed CUDA-event durations
            tot_ms = sum(k["ms"] for k in kern.values())
            match_tflops = FLOP_PER_PAIR * T_loc * D / (tot_ms * 1e-3) / 1e12
            roof_kernel = " + ".join(sorted(kern)) + " (fused tcgen05 xcorr_eff)"
            per_unit, traffic_src = ncu_traffic(args.mode)
            if per_unit:
                roof_traffic = sum(per_unit.get(n, 0.0) * k["units"] for n, k in kern.items())
            roof_extra = {"kernels": {n: {"launches": k["launches"], "avg_ms_per_launch": k["ms"] / k["launches"],
                                          "share_of_match": k["ms"] / match_ms} for n, k in kern.items()}}
        enc_tflops = FLOP_PER_OBJECT * n_enc / (enc_ms * 1e-3) / 1e12
        line = {
            "metric": METRIC, "value": value, "unit": "pairs/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": cfg["scaling"], "vs_baseline": None, "dtype": DTYPE[args.mode],
            "data": "synthetic",
            "config": {"workload": f"{cfg['tag']} encode of {T_loc} tracks/GPU + {D} detections x {NPTS} pts "
                                   f"(backbone_list {list(BLIST)}), {T_loc}x{D} all-pairs xcorr_eff match per GPU"
                                   + (f" = a fixed {T_total}x{D} matrix over {world} rank(s)" if strong_main else ""),
                       "mode": MODE_TEXT[args.mode],
                       "l2": "no flush needed: each step streams >1 GB of activations (>> 126 MB L2)",
                       "sharding": f"track rows over {world} rank(s), one all-gather of detection embeddings"},
            "objects_encoded_per_s": n_enc * world / (enc_ms * 1e-3),
            "phase_ms": {"encode": enc_ms, "match": match_ms},
            "per_step_ms": per_step,
            "gpu_launches": launches,
            "clocks": clocks,
            "e2e": {"value": pairs_total / (e2e_ms / args.steps * 1e-3), "unit": "pairs/s",
                    "h2d_bytes_per_step": (tracks_h.numel() + dets_h.numel()) * 4, "d2h_bytes_per_step": out_h.numel() * 4},
            "roofline": {"bound": "tensor", "achieved": match_tflops, "peak": peak_tf, "unit": "TFLOP/s",
                         "frac": (match_tflops / peak_tf) if match_tflops else None, "traffic": roof_traffic,
                         "traffic_source": traffic_src,
                         "per": "all fused launches of one step (three kernels x both directions x pair chunks), rank 0",
                         "kernel": roof_kernel, "peak_source": pk_src + " bf16 sustained (MEASURED_PEAKS.json)", **roof_extra},
            "encoder": {"bound": "tensor", "objects_per_s": n_enc / (enc_ms * 1e-3), "achieved": enc_tflops, "peak": peak_tf,
                        "unit": "TFLOP/s", "frac": enc_tflops / peak_tf,
                        "per": f"one encode of {n_enc} objects x {NPTS} pts on rank 0 (CUDA-graph replay of the public encode(): device "
                               f"time, not the host's launch rate), {FLOP_PER_OBJECT / 1e6:.0f} MFLOP/object algorithmic"},
        }
        if fast:
            line["fast_mode"] = fast
        if strong:
            line["strong"] = strong
        if not args.no_cpu_baseline and world == 1 and args.config == "c2":
            line["parity"] = parity_block(model, dev)
            line["cpu_baseline"] = cpu_reference_sample()
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
