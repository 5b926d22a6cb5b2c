"""Tick time when only some streams have a frame (BatchedTracker.step(present=...)).

    python benchmarks/bench_presence.py [--steps K] [--warmup W] [--chunks P] [--out FILE]

Workload C3 of bench.py (1024 streams, ~50 detections per frame, nn_budget 100, max_age 60, the same 110-tick pre-roll
with every stream present), then K timed ticks in which a seeded random fraction 0 / 0.25 / 0.5 of the streams has no
frame, drawn anew each tick.  Each camera's own frame sequence advances only on its present ticks, as for a camera
running at a lower frame rate: its next frame continues where its last one left off.  Fraction 0 is run twice: present=None and an all-ones presence tensor.  Each variant
gets its own tracker with the identical pre-roll.  Reported per variant: device ms per tick (CUDA events around K
ticks issued back to back, counts reduced every tick) and present stream-frames per second.  Prints one JSON line.
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import bench  # noqa: E402  (the C3 constants)


def run(frac, mode, args):
    import torch
    from deepdish_b200.batched import BatchedTracker
    from deepdish_b200.scene import Scene, SceneBatch
    dev = torch.device("cuda", 0)
    S, K, W = bench.S_PER_GPU, args.steps, args.warmup
    bt = BatchedTracker(S, bench.LABELS, max_tracks=bench.TMAX, max_dets=bench.DMAX, budget=bench.BUDGET,
                        max_age=bench.MAX_AGE, device=dev, n_chunks=args.chunks)
    scene = Scene(S, bench.N_OBJECTS, bench.DMAX, n_labels=len(bench.LABELS), seed=1234, device=dev)
    for _ in range(bench.PREROLL):
        bt.step(scene.step())
    bt.check()
    frames = [scene.step() for _ in range(W + K)]             # every camera's own frame sequence
    g = torch.Generator(device=dev).manual_seed(7)
    if mode == "none":
        pres = [None] * (W + K)
    else:
        pres = [(torch.rand(S, generator=g, device=dev) >= frac).contiguous() for _ in range(W + K)]
    if frac > 0:
        seq = {k: torch.stack([getattr(b, k) for b in frames]) for k in SceneBatch.__slots__}
        nxt, rows = torch.zeros(S, dtype=torch.long, device=dev), torch.arange(S, device=dev)
        frames = []
        for p in pres:
            frames.append(SceneBatch(*(seq[k][nxt, rows].contiguous() for k in SceneBatch.__slots__)))
            nxt += p.long()
        del seq
    for b, p in zip(frames[:W], pres[:W]):
        bt.step(b, join=False, reduce=True, present=p)
    bt.join()
    torch.cuda.synchronize()
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for b, p in zip(frames[W:], pres[W:]):
        bt.step(b, join=False, reduce=True, present=p)
    bt.join()
    end.record()
    torch.cuda.synchronize()
    ms = start.elapsed_time(end) / K
    bt.check()
    present_frames = S * K if mode == "none" else int(sum(int(p.sum()) for p in pres[W:]))
    out = {"absent_fraction": frac, "present": mode, "ms_per_tick": round(ms, 4),
           "present_stream_frames_per_s": round(present_frames / (K * ms * 1e-3)),
           "present_fraction_measured": round(present_frames / (S * K), 4)}
    del bt, frames
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--chunks", type=int, default=2, help="stream chunks (bench.py's default)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_presence.py measures the B200 path: no CUDA device")
    res = [run(0.0, "none", args), run(0.0, "ones", args), run(0.25, "mask", args), run(0.5, "mask", args)]
    line = json.dumps({"workload": bench.WORKLOAD, "gpu": torch.cuda.get_device_name(0), "steps": args.steps,
                       "warmup": args.warmup, "stream_chunks": args.chunks, "results": res})
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
