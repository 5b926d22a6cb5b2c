"""Cost of the per-tick crossing records (BatchedTracker(crossing_capacity=...), crossings()).

    python benchmarks/bench_events.py [--steps K] [--reps R] [--cap N] [--out FILE]

Workload C3 of bench.py (1024 streams, ~50 detections per frame, nn_budget 100, max_age 60) on two stream chunks, the
same 110-tick pre-roll, on two trackers: records off (crossing_capacity 0) and on (--cap records per chunk and tick).
Both see the same frames in the same order, so their states stay identical.  Then R rounds, alternating off / on, of
K ticks each for:
  - step: device-resident batches, counts reduced every tick; "on" also copies each tick's records to pinned memory
    (out_events_host), "on_device" keeps them on the device;
  - host: step_host_packed with the ids read back every tick; "on" also copies the records.
Reported: the median ms per tick of each variant (CUDA events around K ticks issued back to back), the records per
chunk and tick (mean, max) of the timed "on" ticks, the card name and its power limit.  Prints one JSON line.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import bench  # noqa: E402  (the C3 constants)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [x.strip() for x in q.split(",")]
        return name, power
    except Exception as e:          # no nvidia-smi: the device name from the runtime, the power limit unknown
        import torch
        return torch.cuda.get_device_name(0), "unknown (%r)" % (e,)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--cap", type=int, default=16384, help="crossing records per chunk and tick of the 'on' tracker")
    ap.add_argument("--chunks", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_events.py needs a CUDA device")
    from deepdish_b200.batched import BatchedTracker
    from deepdish_b200.scene import Scene
    dev = torch.device("cuda", 0)
    S, K, R = bench.S_PER_GPU, args.steps, args.reps
    mk = lambda cap: BatchedTracker(S, bench.LABELS, max_tracks=bench.TMAX, max_dets=bench.DMAX, budget=bench.BUDGET,
                                    max_age=bench.MAX_AGE, device=dev, n_chunks=args.chunks, crossing_capacity=cap)
    trk = {"off": mk(0), "on": mk(args.cap)}
    scene = Scene(S, bench.N_OBJECTS, bench.DMAX, n_labels=len(bench.LABELS), seed=1234, device=dev)
    for _ in range(bench.PREROLL):
        b = scene.step()
        for bt in trk.values():
            bt.step(b)
    for bt in trk.values():
        bt.check()
    ids_host = torch.empty((S, bench.DMAX), dtype=torch.int32).pin_memory()
    ev_host = [trk["on"].new_crossings_buffer() for _ in range(K)]
    per_chunk = []

    def timed(fn):
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / K

    def note_records():
        for buf in ev_host:
            blk = buf.numpy().reshape(args.chunks, -1)
            per_chunk.extend(int(x) for x in blk[:, 0])

    ms = {k: [] for k in ("step_off", "step_on_device", "step_on", "host_off", "host_on")}
    for r in range(R + 1):                   # round 0 warms every variant up and is not reported
        frames = [scene.step() for _ in range(K)]
        host = [trk["on"].pack_host(b) for b in frames]          # the two trackers have the same chunks
        res = {}

        def run_step(name, bt, events, device_only=False):
            def go():
                for f, b in enumerate(frames):
                    bt.step(b, join=False, reduce=True, out_events_host=ev_host[f] if events and not device_only else None)
                bt.join()
            res[name] = timed(go)

        def run_host(name, bt, events):
            def go():
                for f, hb in enumerate(host):
                    bt.step_host_packed(hb, ids_host, out_events_host=ev_host[f] if events else None)
                bt.join()
            res[name] = timed(go)

        # the two trackers must see the same frames: the 'on' tracker runs the step window twice per round (with and
        # without the copy) on the device frames, so the 'off' tracker runs it twice as well
        run_step("step_off", trk["off"], False)
        run_step("step_on_device", trk["on"], True, device_only=True)
        run_step("step_off2", trk["off"], False)
        run_step("step_on", trk["on"], True)
        if r > 0:
            note_records()
        run_host("host_off", trk["off"], False)
        run_host("host_on", trk["on"], True)
        if r > 0:
            note_records()
            ms["step_off"].append(statistics.median([res["step_off"], res["step_off2"]]))
            for k in ("step_on_device", "step_on", "host_off", "host_on"):
                ms[k].append(res[k])
        del host
    for bt in trk.values():
        bt.check()
    name, power = card()
    med = {k: round(statistics.median(v), 4) for k, v in ms.items()}
    out = {"bench": "crossing_events", "workload": bench.WORKLOAD_NAME, "streams": S, "stream_chunks": args.chunks,
           "steps_per_run": K, "rounds": R, "event_cap_per_chunk": args.cap,
           "ms_per_tick_median": med,
           "ms_per_tick_runs": {k: [round(x, 4) for x in v] for k, v in ms.items()},
           "step_overhead_ms": round(med["step_on"] - med["step_off"], 4),
           "host_overhead_ms": round(med["host_on"] - med["host_off"], 4),
           "records_per_chunk_tick": {"mean": round(sum(per_chunk) / max(1, len(per_chunk)), 2),
                                      "max": max(per_chunk, default=0), "samples": len(per_chunk)},
           "overflowed": any(x > args.cap for x in per_chunk),
           "gpu": name, "power_limit": power}
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "a") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
