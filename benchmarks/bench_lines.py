"""Cost of several count lines per camera (BatchedTracker(lines=...)).

    python benchmarks/bench_lines.py [--steps K] [--reps R] [--lines 1,2,4,8] [--chunks P] [--out FILE]

Workload C3 of bench.py (1024 streams, ~50 detections per frame, nn_budget 100, max_age 60) on P stream chunks (default
2, as bench.py), one tracker per line count L: L = 1 is the one-line tracker (the reference's default mid-line, `line=`),
L > 1 counts the first L of: the mid-line, the frame's two diagonals, the horizontal mid-line and the vertical and
horizontal quarter lines, the same set for every camera.  Every tracker sees the same frames in the same order (the
110-tick pre-roll, then the timed ticks), so their tracking states stay identical and only the count-line step differs.
Then R rounds of K ticks for each tracker, the order of the trackers rotated from round to round; each run is timed with
CUDA events around K ticks issued back to back (step(), counts reduced every tick, one join at the end).  Reported: the
median ms per tick of each L, its difference to L = 1, every run, the card name and its power limit.  Prints one JSON
line.
"""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import bench  # noqa: E402  (the C3 constants)
from benchmarks.bench_events import card  # noqa: E402

LINE_SET = [(320.0, 0.0, 320.0, 480.0), (0.0, 0.0, 640.0, 480.0), (0.0, 480.0, 640.0, 0.0), (0.0, 240.0, 640.0, 240.0),
            (160.0, 0.0, 160.0, 480.0), (480.0, 0.0, 480.0, 480.0), (0.0, 120.0, 640.0, 120.0),
            (0.0, 360.0, 640.0, 360.0)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--lines", default="1,2,4,8")
    ap.add_argument("--chunks", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    counts = [int(x) for x in args.lines.split(",")]
    if any(not 1 <= n <= len(LINE_SET) for n in counts):
        raise SystemExit("--lines: each count must be within 1..%d" % len(LINE_SET))
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_lines.py needs a CUDA device")
    from deepdish_b200.batched import BatchedTracker
    from deepdish_b200.scene import Scene
    dev = torch.device("cuda", 0)
    S, K, R = bench.S_PER_GPU, args.steps, args.reps

    def make(n):
        kw = dict(line=LINE_SET[0]) if n == 1 else dict(lines=LINE_SET[:n])
        return BatchedTracker(S, bench.LABELS, max_tracks=bench.TMAX, max_dets=bench.DMAX, budget=bench.BUDGET,
                              max_age=bench.MAX_AGE, device=dev, n_chunks=args.chunks, **kw)

    trk = {n: make(n) for n in counts}
    scene = Scene(S, bench.N_OBJECTS, bench.DMAX, n_labels=len(bench.LABELS), seed=1234, device=dev)
    for _ in range(bench.PREROLL):
        b = scene.step()
        for bt in trk.values():
            bt.step(b)
    for bt in trk.values():
        bt.check()

    def timed(bt, frames):
        torch.cuda.synchronize()
        a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for b in frames:
            bt.step(b, join=False, reduce=True)
        bt.join()
        e.record()
        torch.cuda.synchronize()
        return a.elapsed_time(e) / K

    ms = {n: [] for n in counts}
    for r in range(R + 1):                   # round 0 warms every tracker up and is not reported
        frames = [scene.step() for _ in range(K)]
        order = counts[r % len(counts):] + counts[:r % len(counts)]
        for n in order:
            t = timed(trk[n], frames)
            if r > 0:
                ms[n].append(t)
    for bt in trk.values():
        bt.check()
    # the trackers saw the same frames: every line they share counts the same
    ref = trk[counts[0]].total_counts.cpu()
    for n, bt in trk.items():
        tot = bt.total_counts.cpu()
        assert (tot if tot.dim() == 2 else tot[0]).equal(ref if ref.dim() == 2 else ref[0]), n
    name, power = card()
    med = {n: round(statistics.median(v), 4) for n, v in ms.items()}
    base = med.get(1)
    out = {"bench": "count_lines", "workload": bench.WORKLOAD_NAME, "streams": S, "stream_chunks": args.chunks,
           "steps_per_run": K, "rounds": R,
           "ms_per_tick_median": {str(n): v for n, v in med.items()},
           "overhead_vs_one_line_ms": {str(n): round(v - base, 4) for n, v in med.items()} if base is not None else None,
           "ms_per_tick_runs": {str(n): [round(x, 4) for x in v] for n, v in ms.items()},
           "total_counts_line0": trk[counts[0]].total_counts.cpu().reshape(-1, len(bench.LABELS), 4)[0].tolist(),
           "gpu": name, "power_limit": power}
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "a") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
