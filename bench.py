#!/usr/bin/env python
"""bench.py -- tracked stream-frames/s of the batched tracking-by-detection tick on B200.

Workload (BASELINE.json configs[2], "C3"): 1024 concurrent camera streams per GPU x ~50 detections
per frame, 128-d features, nn_budget 100, max_age 60: Tracker.predict + Tracker.update (gating +
gallery cosine + matching cascade + IoU stage + Kalman update + lifecycle) + count-line + count
reduction (+ NCCL all-reduce of the [C,4] counters when N > 1).  A "step" is one tick over all
streams of this rank.  Streams shard across ranks with no data-path collective ("weak" scaling:
1024 streams per GPU).

    python bench.py [--gpus N] [--steps K] [--warmup W]             # CUDA arm
    python bench.py --impl reference [--gpus N] [--steps K] [--warmup W]   # CPU reference arm

Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for the definitions.  --dump-outputs DIR (CUDA arm) also
writes what the last timed step computed to DIR/<name>.npy (float64, see last_step_outputs); the inputs depend only
on the arguments, so two builds run with the same arguments can be compared array for array.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

LABELS = ["person", "bicycle", "car"]
S_PER_GPU = 1024
N_OBJECTS = 50
DMAX = 64
TMAX = 128
BUDGET = 100
MAX_AGE = 60
PREROLL = 110          # setup ticks so galleries reach the budget (SURVEY.md section 8d)
WORKLOAD = ("C3: %d streams/GPU x ~%d dets/frame, 128-d feats, nn_budget %d, max_age %d, "
            "predict+cascade+IoU+Kalman update+countline+count reduce" % (S_PER_GPU, N_OBJECTS, BUDGET, MAX_AGE))
WORKLOAD_NAME = "c3"


def set_workload(name):
    """c3 (default, the configuration the metric is quoted on) or c4, the crowd scene of BASELINE.json
    configs[3]: 4096 streams x 200 dets / frame over 8 GPUs = 512 streams per GPU, up to ~270 tracks."""
    global S_PER_GPU, N_OBJECTS, DMAX, TMAX, WORKLOAD, WORKLOAD_NAME
    WORKLOAD_NAME = name
    if name == "c4":
        S_PER_GPU, N_OBJECTS, DMAX, TMAX = 512, 200, 224, 384
        WORKLOAD = ("C4 crowd: %d streams/GPU x ~%d dets/frame, up to %d tracks/stream, 128-d feats, nn_budget %d, "
                    "max_age %d, predict+cascade+IoU+Kalman update+countline+count reduce"
                    % (S_PER_GPU, N_OBJECTS, TMAX, BUDGET, MAX_AGE))


# ------------------------------------------------------------------------------------------------
# CPU reference arm (the oracle port of the reference's numpy/scipy path; the reference itself is
# pure Python and cannot travel to the GPU box -- see DESIGN.md).  One stream per worker process.
# ------------------------------------------------------------------------------------------------
def _cpu_worker(args):
    seed, preroll, warm, steps, workload = args
    set_workload(workload)
    for k in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[k] = "1"
    import torch
    torch.set_num_threads(1)
    from deepdish_b200.scene import Scene
    from oracle import deepsort as od, countline as oc
    sc = Scene(1, N_OBJECTS, DMAX, n_labels=len(LABELS), seed=seed)
    trk = od.Trkr(od.Metric("cosine", 0.2, BUDGET), 0.7, MAX_AGE, 3)
    cnt = oc.LineCounter(oc.default_line(640, 480), LABELS)
    frames = []
    for _ in range(preroll + warm + steps):
        frames.append(sc.step().stream(0))

    def tick(fr):
        tlwh, conf, lab, feat = fr
        dets = [od.Det(tlwh[i], LABELS[lab[i]], conf[i], feat[i]) for i in range(len(conf))]
        trk.predict()
        trk.update(dets)
        cnt.step(trk)

    for fr in frames[:preroll + warm]:
        tick(fr)
    t0 = time.perf_counter()
    for fr in frames[preroll + warm:]:
        tick(fr)
    return time.perf_counter() - t0


def c1_cpu_port(batches, labels, budget, max_age):
    """cpu_baseline leg of configs.c1: the oracle port of the reference on the same 300 frames, one host core."""
    import torch
    from oracle import deepsort as od
    torch.set_num_threads(1)
    trk = od.Trkr(od.Metric("cosine", 0.2, budget), 0.7, max_age, 3)
    t0 = time.perf_counter()
    n_conf = 0
    for tlwh, conf, lab, feat in batches:
        dets = [od.Det(tlwh[i], labels[lab[i]], conf[i], feat[i]) for i in range(len(conf))]
        trk.predict()
        trk.update(dets)
        n_conf += sum(1 for t in trk.tracks if t.is_confirmed() and t.time_since_update <= 1)
    return time.perf_counter() - t0, [t.track_id for t in trk.tracks], n_conf


def cpu_reference(steps, warm, preroll=100, workers=None):
    import multiprocessing as mp
    cores = workers or os.cpu_count() or 1
    ctx = mp.get_context("spawn")
    with ctx.Pool(cores) as pool:
        times = pool.map(_cpu_worker, [(1000 + i, preroll, warm, steps, WORKLOAD_NAME) for i in range(cores)])
    wall = max(times)
    return {"value": cores * steps / wall, "unit": "stream-frames/s", "cores": cores, "kind": "port",
            "sample": "%d streams (1 per core) x %d frames after %d pre-roll frames, oracle port of the "
                      "reference numpy/scipy path, BLAS threads 1" % (cores, steps, preroll + warm),
            "ms_per_step": 1e3 * wall / steps}


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def stop(self, t0=None, t1=None):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for ts, line in self.rows:
            if t0 is not None and not (t0 - 0.2 <= ts <= t1 + 0.2):
                continue
            p = [x.strip() for x in line.split(",")]
            if len(p) < 9:
                continue
            try:
                sm.append(float(p[1]))
                mx = float(p[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def load_traffic(kernel):
    """DRAM bytes per launch of `kernel` from the committed `ncu --set full` capture (profiles/ncu_traffic.json)."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    try:
        return float(json.load(open(p))[kernel]["dram_bytes_per_launch"])
    except Exception:
        return None


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


DUMP_COV_STREAMS = 64


def last_step_outputs(bt, batch, ids, counts):
    """What a caller of the timed path holds after its last step, as float64 host arrays: the det -> track ids the
    step returned (-1 past each stream's detection count), the counters all_reduce_counts returned, and the tracker's
    per-stream counters and live tracks in track order (id, state, time since update, Kalman mean), padded past each
    stream's track count with track_id -1 and zeros, so that every array is finite.  The Kalman covariances only for
    a fixed, seeded sample of DUMP_COV_STREAMS streams (all of them would be 67 MB at C3)."""
    import numpy as np
    import torch
    S, D = ids.shape
    valid = torch.arange(D, device=ids.device)[None, :] < batch.count.to(ids.device)[:, None]
    out = {"det_track_id": torch.where(valid, ids, -1).cpu().numpy(), "counts": counts.cpu().numpy()}
    v = bt.host_view(["n_tracks", "order", "track_id", "state", "tsu", "mean", "counts"])
    live = np.arange(v["order"].shape[1])[None, :] < v["n_tracks"][:, None]
    slot = np.where(live, v["order"], 0)
    rows = np.arange(S)[:, None]
    for key, name in (("track_id", "track_id"), ("track_state", "state"), ("track_tsu", "tsu")):
        out[key] = np.where(live, v[name][rows, slot], -1)
    out["track_mean"] = np.where(live[..., None], v["mean"][rows, slot], 0.0)
    out["stream_counts"] = v["counts"]
    pick = np.sort(np.random.default_rng(0).choice(S, min(S, DUMP_COV_STREAMS), replace=False))
    cov = bt.host_view(["cov"], streams=pick)["cov"]
    out["track_cov"] = np.where(live[pick][..., None, None], cov[np.arange(len(pick))[:, None], slot[pick]], 0.0)
    out["track_cov_streams"] = pick
    out = {k: np.asarray(a, dtype=np.float64) for k, a in out.items()}
    assert sum(a.nbytes for a in out.values()) <= 64 << 20 and all(np.isfinite(a).all() for a in out.values())
    return out


def gpu_arm(args):
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = None
    if world > 1 and not args.no_affinity:
        # one rank per GPU: run (and allocate the pinned host batches) on the CPUs next to this rank's GPU, so the
        # uploads of 8 ranks do not all cross the socket interconnect
        try:
            import pynvml
            pynvml.nvmlInit()
            pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(local))
            numa = sorted(os.sched_getaffinity(0))
        except Exception as e:            # no NVML / not permitted: leave the scheduler alone
            numa = "unavailable: %r" % (e,)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    from deepdish_b200.batched import BatchedTracker
    from deepdish_b200.scene import Scene
    K, W = args.steps, args.warmup
    S = S_PER_GPU

    # CPU baseline first (rank 0, N=1 only) -- before the GPU is busy, bounded sample
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_reference(steps=60, warm=0, preroll=100)

    P = args.chunks
    knobs = dict(gallery_impl=args.gallery_impl, cosine_ctas_per_sm=args.cosine_ctas, match_warps=args.match_warps,
                 gallery_stages=args.gallery_stages, gallery_waves=args.gallery_waves, gallery_turns=not args.no_turns,
                 engine_graphs=not args.no_graphs)
    bt = BatchedTracker(S, LABELS, max_tracks=TMAX, max_dets=DMAX, budget=BUDGET, max_age=MAX_AGE, device=dev,
                        n_chunks=P, **knobs)
    scene = Scene(S, N_OBJECTS, DMAX, n_labels=len(LABELS), seed=1234 + rank, device=dev)
    pre = [scene.step() for _ in range(PREROLL)]
    for b in pre:
        bt.step(b)
    bt.reduce_counts()
    bt.check()
    frames = [scene.step() for _ in range(W + K)]             # inputs resident in HBM
    e2e_dev = [scene.step() for _ in range(W + K)]
    torch.cuda.synchronize()

    # ---- main timed region: K ticks, stream chunks pipelined, counts reduced (+ NCCL) every tick
    def tick(b):
        ids = bt.step(b, join=False, reduce=True)
        return ids, bt.all_reduce_counts(reduced=True, async_op=True)   # NCCL on its own stream: no rendezvous per tick

    for b in frames[:W]:
        tick(b)
    bt.join()
    bt.wait_counts()
    g0 = int(bt.gallery_vectors().sum())
    conf0 = int(((bt.v["state"] == 2).sum()))
    dets = sum(int(b.count.sum()) for b in frames[W:])
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.25)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    st0 = bt.engine_stats()
    t0 = time.perf_counter()
    start.record()
    for b in frames[W:]:
        last = tick(b)
    enq_ms = 1e3 * (time.perf_counter() - t0)      # host time to issue the K ticks ...
    st1 = bt.engine_stats()
    blocked_ms = st1[2] - st0[2]                   # ... of which blocked in the run-ahead throttle (pool polls: the host
    launches = st1[1] - st0[1]                     #     may not run more than 3 ticks ahead of the device)
    bt.join()
    bt.wait_counts()                               # every count all-reduce of the timed ticks has completed
    end.record()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    clocks = sampler.stop(t0, t1) if rank == 0 else None
    dump = last_step_outputs(bt, frames[-1], *last) if args.dump_outputs and rank == 0 else None
    ms = start.elapsed_time(end)
    state_bytes = bt.memory_bytes()
    # what the gallery kernel must move from HBM for the last tick, read from the work records k_gate wrote for it (one
    # per streamed track: gallery rows, gate-passing detections): every streamed track's half pages ONCE (a track with
    # more than 8 gate-passing detections is streamed again per group of 8, but those passes hit L2), the detections'
    # half rows, one 64-byte work record per track
    g_streamed = q_rows = w_items = 0.0
    for c in bt.chunks:
        n_work = int(c.v["work_ctl"][0])
        rec = c.v["work_rec"][:n_work]
        g_streamed += float(rec[:, 2].sum())
        q_rows += float(rec[:, 3].sum())
        w_items += float(n_work)
    cand_per_track = q_rows / max(1.0, w_items)                         # gate-passing detections per streamed track
    g1 = int(bt.gallery_vectors().sum())
    conf1 = int(((bt.v["state"] == 2).sum()))
    bt.check()

    # ---- end-to-end through the public API with pinned host buffers (same tracker, next K ticks)
    # the host batch is ragged, like the reference's per-stream lists of Detection objects: one pinned blob per
    # stream chunk holding only the detections that exist (BatchedTracker.pack_host)
    host = [bt.pack_host(b) for b in e2e_dev]
    del e2e_dev
    ids_host = torch.empty((S, DMAX), dtype=torch.int32).pin_memory()
    cnt_host = torch.empty((len(LABELS), 4), dtype=torch.int64).pin_memory()
    for hb in host[:W]:
        bt.step_host_packed(hb, ids_host)
    bt.join()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    es, ee = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    st0 = bt.engine_stats()
    tw0 = time.perf_counter()
    es.record()
    for hb in host[W:]:
        cnt = bt.step_host_packed(hb, ids_host)
        cnt = bt.all_reduce_counts(reduced=True)
        cnt_host.copy_(cnt, non_blocking=True)
    e2e_enq_ms = 1e3 * (time.perf_counter() - tw0)
    e2e_blocked_ms = bt.engine_stats()[2] - st0[2]
    bt.join()
    ee.record()
    torch.cuda.synchronize()
    e2e_wall_ms = 1e3 * (time.perf_counter() - tw0)
    e2e_ms = max(es.elapsed_time(ee), e2e_wall_ms)
    bt.check()
    h2d = sum(bt.packed_nbytes(hb) for hb in host[W:]) // K
    d2h = ids_host.numel() * 4 + cnt_host.numel() * 8
    del host

    # ---- per-kernel pass: the same K ticks on a single-stream (n_chunks=1) tracker so that CUDA events
    #      between the kernels measure each kernel alone (rank 0 only; roofline of the dominant kernel)
    stage = [0.0, 0.0, 0.0, 0.0, 0.0]
    single_ms = None
    if rank == 0:
        del bt
        torch.cuda.empty_cache()
        bt1 = BatchedTracker(S, LABELS, max_tracks=TMAX, max_dets=DMAX, budget=BUDGET, max_age=MAX_AGE, device=dev, **knobs)
        for b in pre + frames[:W]:
            bt1.step(b)
        evs = [bt1.new_events(6) for _ in range(K)]
        s1, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        s1.record()
        for i, b in enumerate(frames[W:]):
            bt1.predict()
            bt1.update_profiled(b.tlwh, b.conf, b.label, b.feat, b.count, evs[i])
            bt1.countline()
            bt1.reduce_counts()
        e1.record()
        torch.cuda.synchronize()
        single_ms = s1.elapsed_time(e1)
        for ev in evs:
            for j in range(5):
                stage[j] += bt1.elapsed_ms(ev[j], ev[j + 1]) / K
        bt1.check()
        del bt1
    del pre

    t = torch.tensor([ms, e2e_ms], dtype=torch.float64, device=dev)
    tot = torch.tensor([float(g0 + g1) / 2, float(conf0 + conf1) / 2, float(dets), g_streamed, q_rows, w_items],
                       dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    ms_all, e2e_all = float(t[0]), float(t[1])
    if rank == 0:
        peak, peak_src = load_peaks()
        G, TC = float(tot[0]) / world, float(tot[1]) / world            # per GPU, per tick
        Dn = float(tot[2]) / world / K
        gc_ms = stage[2]
        tick_bytes = 512.0 * (G + Dn + Dn) + 1152.0 * (TC * 1.1) + 44.0 * Dn      # SURVEY 8d B_trk summed over streams
        f32_bytes = 512.0 * G + 512.0 * Dn + 16.0 * TC                            # SURVEY 8d figure for this kernel (f32 rows)
        half = args.gallery_impl != "exact"
        kname = {"default": "k_gallery_stream", "exact": "k_cosine"}[args.gallery_impl]
        traffic = load_traffic(kname) if WORKLOAD_NAME == "c3" else None
        # bytes the kernel MUST move from HBM: the half page rows of every streamed track (once), the detections' half
        # rows and the work records; the exact re-check (a few f32 rows per track) comes on top and is in `traffic`
        Gs, Qr, Wi = (float(tot[k]) / world for k in (3, 4, 5))
        must = (256.0 * Gs + 256.0 * Qr + 64.0 * Wi + 4.0 * Qr) if half else f32_bytes
        achieved = must / (gc_ms * 1e-3) / 1e9
        roof = {"bound": "hbm", "kernel": kname, "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                "bytes_per_launch": must, "ms_per_launch": gc_ms,
                "dram_achieved": (traffic / (gc_ms * 1e-3) / 1e9) if traffic else None,
                "dram_frac": (traffic / (gc_ms * 1e-3) / 1e9 / peak) if traffic else None,
                "f32_equivalent": {"bytes_per_launch": f32_bytes, "achieved": f32_bytes / (gc_ms * 1e-3) / 1e9,
                                   "frac": f32_bytes / (gc_ms * 1e-3) / 1e9 / peak,
                                   "note": "SURVEY 8d counts 512 B per f32 gallery row; the kernel streams the half shadow, "
                                           "so this figure can exceed 1 and is not a physical fraction"},
                "note": ("achieved = bytes the kernel must move (256 B per streamed half gallery row + half query rows + work "
                         "records) / its CUDA-event time in this run; traffic = dram__bytes_read+write of one launch from the "
                         "committed ncu capture (profiles/ncu_traffic.json), dram_frac = traffic / time / peak"
                         if half else "exact f32 gallery pass: 512 B per gallery row"),
                "tick_bytes": tick_bytes, "tick_frac": tick_bytes / (ms_all / K * 1e-3) / 1e9 / peak}
        extras = None
        if world == 1 and not args.no_configs:
            sys.path.insert(0, os.path.join(ROOT, "benchmarks"))
            import configs as extra_configs
            extras = extra_configs.run_all(knobs=knobs, cpu_port=None if args.no_cpu_baseline else c1_cpu_port)
        out = {
            "metric": "tracked stream-frames/s", "value": S * world * K / (ms_all * 1e-3),
            "unit": "stream-frames/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_all / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64 (Kalman/gating/IoU/LSAP/count-line) + f32 (cosine)", "data": "synthetic",
            "config": {"workload": WORKLOAD, "streams_per_gpu": S, "max_tracks": TMAX, "max_dets": DMAX,
                       "preroll_ticks": PREROLL, "stream_chunks": P, "gallery_vectors_per_stream": G / S,
                       "tracker_state_bytes": state_bytes,
                       "confirmed_tracks_per_stream": TC / S, "dets_per_frame": Dn / S, "gate_passing_dets_per_streamed_track": cand_per_track,
                       "l2": "inputs larger than L2: %.2f GB of galleries streamed per tick" % (512 * G / 1e9)},
            "e2e": {"value": S * world * K / (e2e_all * 1e-3), "unit": "stream-frames/s",
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": e2e_all / K,
                    "host_enqueue_ms_per_step": (e2e_enq_ms - e2e_blocked_ms) / K,
                    "host_throttled_ms_per_step": e2e_blocked_ms / K, "rank0_cpu_affinity": numa},
            "host_enqueue_ms_per_step": (enq_ms - blocked_ms) / K,
            "host_throttled_ms_per_step": blocked_ms / K,
            "host_note": "host_enqueue = host time to issue a tick (one call into the native engine: per chunk the prep kernel "
                         "+ the captured graphs of the rest); host_throttled = time the host was additionally BLOCKED because it "
                         "may not run more than 3 ticks ahead of the device (page-pool polls)",
            "gpu_launches": launches,
            "clocks": clocks,
            "roofline": roof,
            "stage_ms": {"pass": "same K ticks, n_chunks=1, CUDA events between kernels", "prep": stage[0],
                         "gate": stage[1], "cosine": stage[2], "match": stage[3], "apply": stage[4],
                         "tick_total_single_stream": single_ms / K, "tick_total_pipelined": ms_all / K},
            "cpu_baseline": cpu,
            "configs": extras,
        }
        if dump is not None:
            import numpy as np
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, a in dump.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = cpu_reference(steps=args.steps, warm=args.warmup, preroll=100)
    out = {"impl": "reference", "metric": "tracked stream-frames/s", "value": r["value"],
           "unit": "stream-frames/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": "f64 (Kalman/gating/IoU/LSAP/count-line) + f32 (cosine)", "data": "synthetic",
           "config": {"workload": WORKLOAD, "sample": r["sample"]},
           "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
           "e2e": {"value": r["value"], "unit": "stream-frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the C1 / C2 / C4 / C5 measurements folded into `configs` (N = 1 only)")
    ap.add_argument("--no-affinity", action="store_true", help="multi-GPU: do not pin each rank to its GPU's CPUs")
    ap.add_argument("--workload", default="c3", choices=["c3", "c4"], help="c3 = the metric's configuration (default)")
    ap.add_argument("--gallery-impl", default="default", choices=["default", "exact"],
                    help="A/B knob: gallery kernel (bit-identical): default (half pre-pass stream), exact f32 pass")
    ap.add_argument("--cosine-ctas", type=int, default=0, help="A/B knob: CTAs per SM of the persistent gallery kernel")
    ap.add_argument("--gallery-stages", type=int, default=0, help="A/B knob: ring stages per warp pair of the default gallery kernel")
    ap.add_argument("--gallery-waves", type=int, default=0, help="A/B knob: 0 = one persistent gallery CTA per SM (default), W = one warp triple per CTA in W waves")
    ap.add_argument("--no-turns", action="store_true", help="A/B knob: chunks do not take turns on the gallery stream")
    ap.add_argument("--no-graphs", action="store_true", help="A/B knob: the engine launches the tick's kernels plainly instead of replaying captured graphs")
    ap.add_argument("--match-warps", type=int, default=0, help="A/B knob: warps per stream in the matching kernel (0 = by size)")
    ap.add_argument("--chunks", type=int, default=2, help="stream chunks pipelined on separate CUDA streams")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy (float64; rank 0's streams)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "cuda":
        ap.error("--dump-outputs needs --impl cuda")
    set_workload(args.workload)
    args.warmup = max(args.warmup, 3) if args.impl == "cuda" else args.warmup
    if args.impl == "reference":
        reference_arm(args)
    else:
        gpu_arm(args)


if __name__ == "__main__":
    main()
