"""Gated linear assignment (kernels.linear_assignment, csrc/assign.cu) against the host alternative (device -> host copy + scipy)
on the same matrices: B in {1, 64} problems at T = D in {64, 256, 1024, 4096}, scores ~ N(0, 1) float32, min_score = -10
(every pair above the threshold), dense or with an 8-class gate.

Device time: CUDA events around the whole public call (output / workspace allocation and the int64 conversion included),
averaged over repeated calls after one warm-up call; inputs stay resident (at B = 1 they fit in L2).
Host time: one D2H copy of the batch (scores + gate), then scipy.optimize.linear_sum_assignment on the T x (D + T) matrix of
tests/assign_reference.py per problem.  At B = 64 and T >= 1024 scipy runs on the first `host_problems_timed` problems only;
`host_ms_per_problem` is what was measured, and no batch total is given for those rows.
Writes one JSON object per shape (and a header line with the GPU name and power limit read in the same run) to --out."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import torch  # noqa: E402

import assign_reference as R  # noqa: E402
from pcreid_b200.kernels import linear_assignment  # noqa: E402

TAU = -10.0
HOST_PROBLEMS = {64: 64, 256: 64, 1024: 4, 4096: 1}     # scipy problems timed per row (at most B)


def gpu_header():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1],
            "torch": torch.__version__, "tau": TAU}


def device_ms(S, mask, budget_s=1.0, max_iters=20):
    linear_assignment(S, TAU, mask)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    linear_assignment(S, TAU, mask)
    e1.record()
    torch.cuda.synchronize()
    first = e0.elapsed_time(e1)
    iters = int(max(1, min(max_iters, budget_s * 1e3 / max(first, 1e-3))))
    e0.record()
    for _ in range(iters):
        linear_assignment(S, TAU, mask)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters, iters


def host(S, mask, n_problems):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    Sh = S.cpu().numpy()
    Mh = None if mask is None else mask.cpu().numpy()
    t1 = time.perf_counter()
    for b in range(n_problems):
        R.assign(Sh[b], TAU, None if Mh is None else Mh[b])
    t2 = time.perf_counter()
    return (t1 - t0) * 1e3, (t2 - t1) * 1e3 / n_problems


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_assign_bench.jsonl"))
    ap.add_argument("--sizes", default="64,256,1024,4096")
    ap.add_argument("--batches", default="1,64")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_assign.py measures the device: it needs a CUDA GPU"
    rows = [gpu_header()]
    print(json.dumps(rows[0]), flush=True)
    for n in (int(x) for x in args.sizes.split(",")):
        for B in (int(x) for x in args.batches.split(",")):
            g = torch.Generator(device="cuda").manual_seed(n + B)
            S = torch.randn((B, n, n), device="cuda", generator=g)
            labels = torch.randint(0, 8, (B, 2, n), device="cuda", generator=g)
            for kind in ("dense", "class8"):
                mask = None if kind == "dense" else labels[:, 0, :, None] == labels[:, 1, None, :]
                dev, iters = device_ms(S, mask)
                k = min(B, HOST_PROBLEMS[n] if n in HOST_PROBLEMS else B)
                d2h, per = host(S, mask, k)
                r = {"B": B, "T": n, "D": n, "gate": kind, "device_ms": round(dev, 4), "device_iters": iters,
                     "d2h_ms": round(d2h, 3), "host_problems_timed": k, "host_ms_per_problem": round(per, 3),
                     "host_ms_batch": round(d2h + per * B, 3) if k == B else None}
                if r["host_ms_batch"] is not None:
                    r["device_speedup"] = round(r["host_ms_batch"] / dev, 2)
                rows.append(r)
                print(json.dumps(r), flush=True)
            del S, labels
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        for r in rows:
            f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
