"""Device time of the count-line kernel alone (k_countline), crossing records off and on.

    python benchmarks/bench_countline.py [--steps K] [--reps R] [--lines L] [--cap N] [--out FILE]

Workload C3 of bench.py (1024 streams, ~50 detections per frame, nn_budget 100, max_age 60) on one stream chunk, two
trackers: records off (crossing_capacity 0) and on (--cap records per tick), counting the reference's mid-line (L = 1,
`line=`) or the first L lines of benchmarks/bench_lines.py's set.  Every tick is issued call by call -- predict(),
update(), countline() -- so that the count-line kernel runs on its own.  Both trackers see the same frames in the same
order (the 110-tick pre-roll, then R rounds of K ticks, the order of the trackers swapped every round), so their states
stay identical.  Each round runs under torch.profiler (CUDA activity only) and the kernel's durations are read from
its trace.  Reported: the median, quartiles and extremes of the kernel's duration per tracker, the summed counters
(equal in both, and equal from one build to the next), the card name and its power limit.  Prints one JSON line.
"""
import argparse
import json
import os
import statistics
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import bench  # noqa: E402  (the C3 constants)
from benchmarks.bench_events import card  # noqa: E402
from benchmarks.bench_lines import LINE_SET  # noqa: E402


def kernel_us(prof, name):
    """Durations (us) of the kernels whose name contains `name`, in launch order, from the profiler's trace."""
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as fh:
            ev = json.load(fh)["traceEvents"]
    ks = [e for e in ev if e.get("cat") == "kernel" and name in e.get("name", "")]
    return [float(e["dur"]) for e in sorted(ks, key=lambda e: e["ts"])]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--reps", type=int, default=4)
    ap.add_argument("--lines", type=int, default=1)
    ap.add_argument("--cap", type=int, default=16384, help="crossing records per tick of the 'on' tracker")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not 1 <= args.lines <= len(LINE_SET):
        raise SystemExit("--lines: within 1..%d" % len(LINE_SET))
    import torch
    from torch.profiler import profile, ProfilerActivity
    if not torch.cuda.is_available():
        raise SystemExit("bench_countline.py needs a CUDA device")
    from deepdish_b200.batched import BatchedTracker
    from deepdish_b200.scene import Scene
    dev = torch.device("cuda", 0)
    S, K, R = bench.S_PER_GPU, args.steps, args.reps
    kw = dict(line=LINE_SET[0]) if args.lines == 1 else dict(lines=LINE_SET[:args.lines])
    mk = lambda cap: BatchedTracker(S, bench.LABELS, max_tracks=bench.TMAX, max_dets=bench.DMAX, budget=bench.BUDGET,
                                    max_age=bench.MAX_AGE, device=dev, crossing_capacity=cap, **kw)
    trk = {"off": mk(0), "on": mk(args.cap)}
    scene = Scene(S, bench.N_OBJECTS, bench.DMAX, n_labels=len(bench.LABELS), seed=1234, device=dev)

    def tick(bt, b):
        bt.predict()
        bt.update(b.tlwh, b.conf, b.label, b.feat, b.count)
        bt.countline()

    for _ in range(bench.PREROLL):
        b = scene.step()
        for bt in trk.values():
            tick(bt, b)
    for bt in trk.values():
        bt.check()
    us = {k: [] for k in trk}
    names = list(trk)
    for r in range(R + 1):                   # round 0 warms both trackers up and is not reported
        frames = [scene.step() for _ in range(K)]
        order = names if r % 2 == 0 else names[::-1]
        for n in order:
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for b in frames:
                    tick(trk[n], b)
                torch.cuda.synchronize()
            if r > 0:
                us[n] += kernel_us(prof, "k_countline")
    for bt in trk.values():
        bt.check()
    counts = {n: bt.reduce_counts().cpu().tolist() for n, bt in trk.items()}
    assert counts["off"] == counts["on"]

    def summary(v):
        q = statistics.quantiles(v, n=4)
        return {"median": round(statistics.median(v), 3), "q1": round(q[0], 3), "q3": round(q[2], 3),
                "min": round(min(v), 3), "max": round(max(v), 3), "n": len(v)}

    name, power = card()
    out = {"bench": "countline_kernel", "workload": bench.WORKLOAD_NAME, "streams": S, "lines": args.lines,
           "steps_per_round": K, "rounds": R, "unit": "us",
           "records_off": summary(us["off"]), "records_on": summary(us["on"]),
           "total_counts": counts["off"], "gpu": name, "power_limit": power}
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "a") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
