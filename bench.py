#!/usr/bin/env python
"""bench.py — benchmarks of the detect+track hot path (contract: see the task prompt / DESIGN.md §6).

    python bench.py --gpus N --steps K --warmup W            # our arm (CUDA, one process per GPU)
    python bench.py --impl reference --gpus N --steps K ...   # the reference's CPU path (oracle restatement)

Workloads (BASELINE.json `configs`; the default is the headline, configs[2]):
    detect_track30  1024 x 640x480 per GPU: ccv.grayscale + ccv.detect_objects(interval 5, min_neighbors 1),
                    facetrackr's VJ->CS hand-off, then 30 camshift track() calls on the frame          (configs[2])
    detect          the same batch, detection only                                                     (configs[1])
    detect720       512 x 1280x720 per GPU (4096 over 8 GPUs), --interval 3 ("4 scales per octave") or 5 (configs[3])
    streams         --streams S independent 640x480 video streams per GPU (default 1: one per GPU), one frame per
                    stream per call through ht_stream_step: detect until found, then one track() per frame,
                    re-detect when the face is lost; steady-state frames/s                             (configs[4])
`--width/--height/--batch/--interval` override the workload's defaults (e.g. the 320x240 line).

A "step" is one pass of the hot path over one batch (streams: --stream-frames consecutive frames of every stream).
`value` is whole-job frames/s with the batch resident in HBM; `e2e` is the same work through the C ABI on pinned
HOST frames (H2D + D2H inside the timed region).

--dump-outputs DIR writes what the last timed step returned as DIR/<name>.npy (float64, frame or stream index first;
rank 0's share with --gpus > 1), plus frame_index.npy naming the frames the files hold.  The inputs depend only on the
arguments, so two builds of the library can be compared output for output.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.dont_write_bytecode = True      # the tree may be read-only: the benchmark leaves no bytecode caches in it
sys.path.insert(0, str(ROOT))

from headtrackr_b200 import synth  # noqa: E402

N_UNIQUE = 64          # distinct synthetic frames generated on the CPU; the batch tiles them with x-rolls
HBM_PEAK_FALLBACK = 6650.0
WORKLOADS = {
    "detect_track30": dict(width=640, height=480, batch=1024, interval=5, track_calls=30,
                           metric="frames/sec @640x480 (detect+CAMShift)"),
    "detect": dict(width=640, height=480, batch=1024, interval=5, track_calls=0,
                   metric="frames/sec @640x480 (detect)"),
    "detect720": dict(width=1280, height=720, batch=512, interval=3, track_calls=0,
                      metric="frames/sec @1280x720 (detect)"),
    "streams": dict(width=640, height=480, batch=1, interval=5, track_calls=1,
                    metric="frames/sec @640x480 (video streams: detect -> track -> redetect)"),
}


def make_base_frames(W, H, start, n=N_UNIQUE):
    with ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1)) as ex:
        frames = list(ex.map(lambda i: synth.frame(start + i, W, H), range(n)))
    return np.stack(frames)


def stream_frames(seed, W, H, T):
    """One synthetic video stream (SURVEY 8d config 5): the face of frame `seed` drifts 3 px / 2 px per frame; for
    5 frames near the end the face is gone (blurred-noise background only) and then comes back, so that a step also
    contains a lost face and a re-detection.  Returns (T, H, W, 4) u8."""
    base = synth.frame(seed, W, H, n_faces=1)
    empty = synth.frame(seed + 7919, W, H, n_faces=0)
    gone = range(T - 20, T - 15) if T >= 40 else range(0)
    return np.stack([np.roll(empty if t in gone else base, (2 * t, 3 * t), axis=(0, 1)) for t in range(T)])


def measured_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return HBM_PEAK_FALLBACK, "fallback (B200_PROFILING.md 6.65 TB/s)"


def captured_traffic(W, H):
    """dram__bytes_read + dram__bytes_write of k_cascade per frame from this round's committed ncu capture
    (profiles/r02_cascade_dram.json, written by tools/ncu_dram.py from the .ncu-rep) - None when there is no capture
    for this frame size.  Never a constant in this file."""
    p = ROOT / "profiles" / "r02_cascade_dram.json"
    try:
        d = json.loads(p.read_text())
        if (d["width"], d["height"]) == (W, H):
            return float(d["dram_bytes_per_frame"]), d.get("source", str(p.name))
    except Exception:
        pass
    return None, None


DUMP_LIMIT = 64 << 20       # bytes --dump-outputs may write in all


def step_outputs(workload, rects, counts, found, objs, wins, events):
    """The records one step of `workload` returns, decoded from the C structs (include/headtrackr_b200.h) into float64
    arrays with the frame (streams: stream) index first.  Rect rows past a frame's count hold no result and are zeroed."""
    if workload == "streams":
        ev = events.cpu().numpy()                       # (T, B, 56) ht_stream_event
        dec = np.concatenate([ev.view(np.int32)[..., :2].astype(np.float64), ev.view(np.float64)[..., 1:7]], axis=-1)
        return {"events": dec.transpose(1, 0, 2)}       # detection, status, x, y, width, height, angle, confidence
    n = counts.cpu().numpy()
    r = rects.cpu().numpy()                             # (B, K, 6) ht_rect
    r = np.concatenate([r[..., :5], r.view(np.int32)[..., 10:11].astype(np.float64)], axis=-1)  # ..., confidence, neighbors
    r[np.arange(r.shape[1])[None, :] >= n[:, None]] = 0.0
    out = {"rects": r, "counts": n.astype(np.float64)}
    if workload == "detect_track30":
        o = objs.cpu().numpy()                          # (B, 6) int32 = ht_trackobj: x, y, width, height, fp64 angle
        out.update(found=found.cpu().numpy().astype(np.float64),
                   objs=np.concatenate([o[:, :4].astype(np.float64), np.ascontiguousarray(o[:, 4:6]).view(np.float64)], axis=1),
                   windows=wins.cpu().numpy().astype(np.float64))
    return out


def write_outputs(out_dir, arrays, limit=DUMP_LIMIT):
    """DIR/<name>.npy for every array and DIR/frame_index.npy, the frames they hold: all of them, or a fixed, seeded
    sample when all of them would exceed `limit` bytes."""
    n = len(next(iter(arrays.values())))
    per_frame = sum(a[0].nbytes for a in arrays.values()) + 8
    room = limit - 128 * (len(arrays) + 1)              # .npy headers
    keep = np.arange(n)
    if n * per_frame > room:
        keep = np.sort(np.random.default_rng(0).choice(n, room // per_frame, replace=False))
    out_dir = Path(out_dir)
    out_dir.mkdir(parents=True, exist_ok=True)
    np.save(out_dir / "frame_index.npy", keep.astype(np.float64))
    for name, a in arrays.items():
        np.save(out_dir / f"{name}.npy", np.ascontiguousarray(a[keep]))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "samples": len(sm),
                "reasons": sorted(reasons)}


def bind_to_gpu_numa_node(local):
    """Pin this rank's host threads (and, by first touch, its pinned staging buffers) to the NUMA node of its GPU:
    eight ranks pushing 1.26 GB per step each over PCIe from the wrong socket cost the 8-GPU e2e line 10 % in round 1."""
    try:
        import torch
        p = torch.cuda.get_device_properties(local)
        bdf = f"{p.pci_domain_id:04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
        node = int(Path(f"/sys/bus/pci/devices/{bdf}/numa_node").read_text())
        if node < 0:
            return {"node": None, "why": "sysfs reports no NUMA node for the GPU"}
        cpus = set()
        for part in Path(f"/sys/devices/system/node/node{node}/cpulist").read_text().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        allowed = cpus & set(os.sched_getaffinity(0))
        if not allowed:
            return {"node": node, "why": "no allowed CPU on that node"}
        os.sched_setaffinity(0, allowed)
        return {"node": node, "cpus": len(allowed), "gpu": bdf}
    except Exception as e:   # never fatal: the numbers are still valid, just not NUMA-local
        return {"node": None, "why": f"{type(e).__name__}: {e}"}


# ------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the CPU oracle (C restatement of src/ccv.js + src/camshift.js)

def cpu_stream(frames, blob, interval):
    """facetrackr's loop (src/facetrackr.js:67-126 + the lost-face rule of src/main.js:230-244, whitebalancing off)
    over one stream on the C oracle.  Returns the number of frames processed."""
    import oracle
    mode, tracker = "VJ", None
    for f in frames:
        if mode == "VJ":
            cand = None
            for r in oracle.detect(f, blob, interval, 1):
                if cand is None or r[4] > cand[4]:
                    cand = r
            if cand is not None and cand[4] > -10:
                tracker = oracle.CamshiftTracker(calc_angles=False)
                tracker.init_tracker(f, *[int(math.floor(v)) for v in cand[:4]])
                mode = "CS"
        else:
            tracker.track(f)
            o = tracker.track_obj()
            if o["width"] == 0 or o["height"] == 0:
                mode = "VJ"
    return len(frames)


def cpu_step(cfg, frames, blob, threads, keep=None):
    import oracle

    def one(i):   # one C call per frame (the GIL is released for its whole duration)
        if cfg["workload"] == "streams":
            return cpu_stream(frames[i], blob, cfg["interval"])
        if cfg["track_calls"] > 0:
            n, found, obj = oracle.detect_track(frames[i], blob, cfg["interval"], 1, False, cfg["track_calls"])
            return (n, found, obj["x"], obj["y"], obj["width"], obj["height"])
        return (len(oracle.detect(frames[i], blob, cfg["interval"], 1)),)

    t0 = time.perf_counter()
    with ThreadPoolExecutor(max_workers=threads) as ex:   # ctypes releases the GIL inside the C oracle
        results = list(ex.map(one, range(len(frames))))
    if keep is not None:
        keep[:] = results       # what the oracle computed for these frames (the GPU arm checks its own batch against it)
    return time.perf_counter() - t0


def usable_cores():
    """Host cores this process may actually use: CPU affinity, capped by a cgroup CPU quota if there is one
    (os.cpu_count() reports the machine, not the container)."""
    try:
        n = len(os.sched_getaffinity(0))
    except (AttributeError, OSError):
        n = os.cpu_count() or 1
    quota = None
    try:
        q, p = Path("/sys/fs/cgroup/cpu.max").read_text().split()[:2]          # cgroup v2
        if q != "max":
            quota = float(q) / float(p)
    except (OSError, ValueError):
        try:
            q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())           # cgroup v1
            p = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0 and p > 0:
                quota = q / p
        except (OSError, ValueError):
            pass
    if quota is not None:
        n = max(1, min(n, int(quota + 0.999)))
    return n


def cpu_sample_frames(cfg, n_sample):
    W, H = cfg["width"], cfg["height"]
    if cfg["workload"] == "streams":
        T = min(cfg["stream_frames"], 40)
        return [stream_frames(1000 + s, W, H, T) for s in range(n_sample)], n_sample * T
    return make_base_frames(W, H, 0, n_sample), n_sample


def cpu_baseline(cfg, n_sample, blob, steps=1, warmup=0, frames=None, keep=None):
    import oracle
    oracle.lib()
    threads = usable_cores()
    if frames is None:
        frames, units = cpu_sample_frames(cfg, n_sample)
    else:
        units = len(frames)
    for _ in range(warmup):
        cpu_step(cfg, frames, blob, threads)
    times = [cpu_step(cfg, frames, blob, threads, keep) for _ in range(steps)]
    total = sum(times)
    what = (f"{len(frames)} synthetic streams x {units // max(len(frames), 1)} frames per step" if cfg["workload"] == "streams"
            else f"{units} of the bench's synthetic frames per step")
    return {"value": units * steps / total, "unit": "frames/s", "cores": threads, "host_cpu_count": os.cpu_count(),
            "kind": "port",
            "sample": f"{what}, C restatement of the reference JS (oracle/ht_oracle.c, -O2, one thread per host core; "
                      f"not V8: no JS engine exists in this image)"}, total / steps


def config_dict(cfg, world, frames_per_gpu_per_step):
    """Same keys in both arms (the driver compares them)."""
    d = {"workload": cfg["workload"], "frame": f"{cfg['width']}x{cfg['height']}", "interval": cfg["interval"],
         "min_neighbors": 1, "track_calls_per_frame": cfg["track_calls"], "sharding": f"frames dp{world}",
         "frames_per_gpu_per_step": frames_per_gpu_per_step}
    if cfg["workload"] == "streams":
        d.update(streams_per_gpu=cfg["batch"], frames_per_stream_per_step=cfg["stream_frames"],
                 sharding=f"streams dp{world}")
    return d


def run_reference(args, cfg):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    blob = synth.load_cascade_blob()
    cb, sec_per_step = cpu_baseline(cfg, args.cpu_sample, blob, steps=args.steps, warmup=args.warmup)
    per_step = args.cpu_sample * (min(cfg["stream_frames"], 40) if cfg["workload"] == "streams" else 1)
    line = {"impl": "reference", "metric": cfg["metric"], "value": cb["value"],
            "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": sec_per_step * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8+f64", "data": "synthetic",
            "config": dict(config_dict(cfg, args.gpus, cfg["batch"] * (cfg["stream_frames"] if cfg["workload"] == "streams" else 1)),
                           reference_sample_frames_per_step=per_step),
            "cpu_baseline": cb,
            "e2e": {"value": cb["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------

def run_ours(args, cfg):
    import torch
    import torch.distributed as dist
    from headtrackr_b200 import Context
    from headtrackr_b200.parallel import agreed

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; this benchmark has no CPU fallback (use --impl reference)")
    torch.cuda.set_device(local)
    numa = bind_to_gpu_numa_node(local) if world > 1 else {"node": None, "why": "single rank"}
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        import datetime
        # a collective that never completes (a rank that died, mismatched calls) aborts the job after 3 minutes instead of
        # hanging it: every collective of this script finishes in milliseconds
        dist.init_process_group("nccl", device_id=torch.device("cuda", local), timeout=datetime.timedelta(seconds=180))
    W, H, B, interval, track_calls = cfg["width"], cfg["height"], cfg["batch"], cfg["interval"], cfg["track_calls"]
    workload = cfg["workload"]
    streams = workload == "streams"
    T = cfg["stream_frames"] if streams else 1
    # per-rank data: independent frames / streams per GPU (weak scaling, frames are the shard unit)
    if streams:
        hv_src = np.stack([stream_frames(rank * 100000 + s, W, H, T) for s in range(B)], axis=1)   # (T, B, H, W, 4)
        host = torch.empty((T, B, H, W, 4), dtype=torch.uint8, pin_memory=True)
        host.numpy()[...] = hv_src
    else:
        base = make_base_frames(W, H, rank * 100000, N_UNIQUE)
        host = torch.empty((B, H, W, 4), dtype=torch.uint8, pin_memory=True)
        hv = host.numpy()
        for j in range(B):
            hv[j] = np.roll(base[j % N_UNIQUE], (j // N_UNIQUE) * 16, axis=1)
    dev = host.cuda(non_blocking=False)
    # a real (non-NULL) stream: the context launches on it, the events time it.  HT_BENCH_STREAM_PRIO: CUDA priority of
    # that stream (torch clamps it to the device's range); the library's background tracking runs below it (HT_PIPE_BG)
    stream = torch.cuda.Stream(priority=int(os.environ.get("HT_BENCH_STREAM_PRIO", "0")))
    torch.cuda.set_stream(stream)
    ctx = Context(max_width=W, max_height=H, max_frames=B, device=local, stream=stream.cuda_stream)
    K = ctx.K
    # Pipelined steps (ht_set_pipeline, default for the detect+track workload): the tracking of step s stays on the
    # library's second stream and runs under the detection of step s+1.  Two output sets alternate so that the records of
    # step s-1 can be gathered while step s is in flight; the last step is joined inside the timed region.
    pipe = bool(args.pipeline) and workload == "detect_track30"
    n_sets = 2 if pipe else 1
    d_rects = [torch.zeros((B, K, 6), dtype=torch.float64, device="cuda") for _ in range(n_sets)]      # ht_rect = 48 B
    d_counts = [torch.zeros((B,), dtype=torch.int32, device="cuda") for _ in range(n_sets)]
    d_found = [torch.zeros((B,), dtype=torch.int32, device="cuda") for _ in range(n_sets)]
    d_objs = [torch.zeros((B, 6), dtype=torch.int32, device="cuda") for _ in range(n_sets)]            # ht_trackobj = 24 B
    d_wins = [torch.zeros((B, 4), dtype=torch.int32, device="cuda") for _ in range(n_sets)]
    d_events = torch.zeros((T, B, 56), dtype=torch.uint8, device="cuda")      # ht_stream_event = 56 B
    # the record every rank contributes to the result gather: one fixed-size row per frame (per stream and frame)
    if workload in ("detect", "detect720"):
        rec_srcs, rec_shape, rec_dtype = d_counts, (B,), torch.int32
    elif streams:
        rec_srcs, rec_shape, rec_dtype = [d_events], (T, B, 56), torch.uint8
    else:
        rec_srcs, rec_shape, rec_dtype = d_objs, (B, 6), torch.int32
    # The gather is double-buffered and runs on its own stream: the records of step s are copied aside and gathered
    # over NCCL while step s+1 is computing, so a slow rank no longer stalls the others on every step.
    gathered = [torch.zeros((world,) + rec_shape, dtype=rec_dtype, device="cuda") for _ in range(2)] if world > 1 else None
    staged = [torch.zeros(rec_shape, dtype=rec_dtype, device="cuda") for _ in range(2)] if world > 1 else None
    comm_stream = torch.cuda.Stream() if world > 1 else None
    gather_events = []
    step_no = [0]
    gather_no = [0]
    ungathered = [None]         # (pipelined) output set whose records have not been gathered yet

    def compute(o=0):
        if workload in ("detect", "detect720"):
            ctx.detect_raw(dev, interval, 1, out_rects=d_rects[0], out_counts=d_counts[0])
        elif streams:
            for t in range(T):
                ctx.stream_step(dev[t], interval, 1, calc_angles=False, out_events=d_events[t])
        else:
            ctx.detect_track(dev, interval, 1, calc_angles=False, n_calls=track_calls,
                             outputs=(d_rects[o], d_counts[o], d_found[o], d_objs[o], d_wins[o]))

    pending = [None, None]      # completion event of the gather that last used staging buffer b

    def gather(src, time_gather=False):
        # the only collective: fixed-size result records gathered over NCCL/NVLink
        b = gather_no[0] & 1
        gather_no[0] += 1
        if pending[b] is not None:
            stream.wait_event(pending[b])        # staged[b] / gathered[b] are free again
        staged[b].copy_(src, non_blocking=True)
        done = torch.cuda.Event()
        done.record(stream)
        comm_stream.wait_event(done)
        with torch.cuda.stream(comm_stream):
            if time_gather:
                g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                g0.record(comm_stream)
            dist.all_gather_into_tensor(gathered[b], staged[b])
            if time_gather:
                g1.record(comm_stream)
                gather_events.append((g0, g1))
            fin = torch.cuda.Event()
            fin.record(comm_stream)
        pending[b] = fin

    def step(time_gather=False):
        o = step_no[0] % n_sets
        compute(o)
        if world > 1:
            if not pipe:
                gather(rec_srcs[0], time_gather)
            else:
                # everything enqueued after compute() is ordered behind the tracking of the PREVIOUS step (the library
                # makes k_group of this step wait for it): its records are complete, and this step writes the other set
                if ungathered[0] is not None:
                    gather(rec_srcs[ungathered[0]], time_gather)
                ungathered[0] = o
        step_no[0] += 1

    def last_outputs():
        o = (step_no[0] - 1) % n_sets
        return d_rects[o], d_counts[o], d_found[o], d_objs[o], d_wins[o]

    def drain():
        if workload == "detect_track30":
            ctx.join()          # the context's stream waits for a pipelined step's tracking (no host wait; no-op otherwise)
        if pipe and world > 1 and ungathered[0] is not None:
            gather(rec_srcs[ungathered[0]], True)
            ungathered[0] = None
        for e in pending:
            if e is not None:
                stream.wait_event(e)

    def barrier():
        drain()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    step_guarded = step

    # Headline = strict: every mean-shift pass of every track() call is summed on the device, as the reference does.
    # The library's default additionally re-uses the moments of windows it has already summed within a launch
    # (ht_set_track_memo, DESIGN.md §5.2) - identical results, far fewer passes when 30 calls hit one frame; that
    # mode is measured separately below and reported under "memo", never as the headline.
    ctx.set_track_memo(False)
    ctx.set_pipeline(pipe)
    if streams:
        ctx.stream_reset(0, B)
    # nvidia-smi needs a few hundred ms before its first sample: start it before the warm-up so that it is sampling
    # every 20 ms when the timed region begins (a short run used to end before the first sample)
    sampler = ClockSampler(local)
    sampler.start()
    t_w = time.perf_counter()
    for _ in range(args.warmup):
        step_guarded()
    barrier()
    # (extra warm-up steps until nvidia-smi is sampling; not timed.)  The decision to run another one is COLLECTIVE:
    # every rank reads its own clock, and a rank that left this loop one iteration before the others would pair its next
    # all_gather with their barrier - a mismatch on the communicator, i.e. a hang.  Rank 0 decides for everybody.
    while agreed(time.perf_counter() - t_w < 0.6, device="cuda"):
        step_guarded()
        barrier()
    l0 = ctx.launch_count
    ctx.profile(True)
    ctx.profile_read(reset=True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record(stream)
    for _ in range(args.steps):
        step_guarded(time_gather=True)
    drain()                     # the last gathers are part of the job
    e1.record(stream)
    barrier()
    ms_local = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:     # before the measurements below reuse the output buffers
        write_outputs(args.dump_outputs, step_outputs(workload, *last_outputs(), d_events))
    prof = ctx.profile_read(reset=True)
    ctx.profile(False)
    track_stats = ctx.debug_track_stats(reset=True)
    launches = ctx.launch_count - l0
    clocks = sampler.stop()
    gather_ms = float(np.mean([a.elapsed_time(b) for a, b in gather_events])) if gather_events else None
    ms = ms_local
    if world > 1:
        t = torch.tensor([ms_local], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    frames_per_step = B * T
    value = world * frames_per_step * args.steps / (ms / 1e3)

    # ---- multi-GPU correctness (SURVEY 4): what rank 0 received from rank r equals what ONE GPU computes for
    #      rank r's frames - rank 0 regenerates the first frames of every other rank and runs them itself ----
    shard_check = None
    if world > 1 and not streams:
        g = gathered[(gather_no[0] - 1) & 1]
        torch.cuda.synchronize()
        if rank == 0:
            n_chk, bad = 8, 0
            for r in range(1, world):
                fr = torch.from_numpy(make_base_frames(W, H, r * 100000, n_chk)).cuda()
                if workload == "detect_track30":
                    _, _, objs, _ = ctx.detect_track(fr, interval, 1, calc_angles=False, n_calls=track_calls)
                    mine = [(o["x"], o["y"], o["width"], o["height"]) for o in objs]
                    theirs = [tuple(int(v) for v in g[r, i, :4].tolist()) for i in range(n_chk)]
                else:
                    _, cnt = ctx.detect_raw(fr, interval, 1)
                    mine = [int(c) for c in cnt]
                    theirs = [int(v) for v in g[r, :n_chk].tolist()]
                bad += sum(1 for a, b in zip(mine, theirs) if a != b)
            shard_check = {"ranks_checked": world - 1, "frames_per_rank": n_chk, "mismatches": bad}
            if bad:
                raise SystemExit(f"bench.py: gathered records differ from a single-GPU run ({bad} frames)")
        dist.barrier()

    # ---- e2e: same work through the public C ABI on pinned HOST frames ----
    h_rects = torch.empty((B, K, 6), dtype=torch.float64, pin_memory=True)
    h_counts = torch.empty((B,), dtype=torch.int32, pin_memory=True)
    h_found = torch.empty((B,), dtype=torch.int32, pin_memory=True)
    h_objs = torch.empty((B, 6), dtype=torch.int32, pin_memory=True)
    h_wins = torch.empty((B, 4), dtype=torch.int32, pin_memory=True)
    h_events = torch.empty((B, 56), dtype=torch.uint8, pin_memory=True)
    L = ctx._L

    def e2e_step():
        if workload in ("detect", "detect720"):
            rc = L.ht_detect(ctx._h, host.data_ptr(), B, W, H, interval, 1, h_rects.data_ptr(), h_counts.data_ptr())
            ctx._check(rc)
        elif streams:
            for t in range(T):   # one blocking call per video frame: upload, kernels, event records back
                ctx._check(L.ht_stream_step(ctx._h, host[t].data_ptr(), B, W, H, interval, 1, 0, h_events.data_ptr()))
        else:
            rc = L.ht_detect_track(ctx._h, host.data_ptr(), B, W, H, interval, 1, 0, track_calls, h_rects.data_ptr(),
                                   h_counts.data_ptr(), h_found.data_ptr(), h_objs.data_ptr(), h_wins.data_ptr())
            ctx._check(rc)

    def timed_e2e():
        if streams:
            ctx.stream_reset(0, B)
        e2e_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            e2e_step()          # returns after the D2H of the results has completed
        barrier()
        s = time.perf_counter() - t0
        if world > 1:
            tt = torch.tensor([s], dtype=torch.float64, device="cuda")
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            s = float(tt.item())
        return s

    e2e_s = timed_e2e()
    e2e_value = world * frames_per_step * args.steps / e2e_s

    # ---- the same steps in the OTHER mode (pipelined <-> every step joins its own tracking), reported beside the headline.
    #      Pipelined as the secondary measurement only on one GPU: the multi-GPU lines stay on the path every earlier
    #      round measured (and the driver's scaling curve compares like with like) ----
    other_mode = None
    if workload == "detect_track30" and (pipe or world == 1):
        try:
            ctx.set_pipeline(not pipe)
            step_guarded()
            barrier()
            ctx.profile(True)
            ctx.profile_read(reset=True)
            u0, u1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            u0.record(stream)
            for _ in range(args.steps):
                step_guarded()
            drain()
            u1.record(stream)
            barrier()
            u_ms = u0.elapsed_time(u1)
            u_prof = ctx.profile_read(reset=True)
            ctx.profile(False)
            if world > 1:
                t = torch.tensor([u_ms], dtype=torch.float64, device="cuda")
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                u_ms = float(t.item())
            other_mode = {"value": world * frames_per_step * args.steps / (u_ms / 1e3), "ms_per_step": u_ms / args.steps,
                          "kernel_ms_per_step": {k: round(v[0] / args.steps, 4) for k, v in u_prof.items()},
                          "note": ("ht_set_pipeline off: the tracking of a step completes before the next step's detection starts"
                                   if pipe else
                                   "ht_set_pipeline on: the tracking of step s runs on the library's second stream under the detection "
                                   "of step s+1 (identical results; the last step is joined inside the timed region; per-kernel times "
                                   "include the waits for SM slots that the overlap causes)")}
        except Exception as e:   # the secondary figure must never cost the headline line
            other_mode = {"error": f"{type(e).__name__}: {e}"}
        ctx.set_pipeline(pipe)

    # ---- library default (window memo on): same steps, device-resident and e2e ----
    memo = None
    if workload == "detect_track30":
        ctx.set_track_memo(True)
        step_guarded()
        barrier()
        ctx.debug_track_stats(reset=True)
        ctx.profile(True)
        ctx.profile_read(reset=True)
        m0, m1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        m0.record(stream)
        for _ in range(args.steps):
            step_guarded()
        drain()
        m1.record(stream)
        barrier()
        memo_ms = m0.elapsed_time(m1)
        memo_prof = ctx.profile_read(reset=True)
        ctx.profile(False)
        memo_stats = ctx.debug_track_stats(reset=True)
        memo_e2e_s = timed_e2e()
        if world > 1:
            t = torch.tensor([memo_ms], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            memo_ms = float(t[0].item())
        memo = {"value": world * B * args.steps / (memo_ms / 1e3), "ms_per_step": memo_ms / args.steps,
                "e2e_value": world * B * args.steps / memo_e2e_s,
                "track_ms_per_step": round(memo_prof["track"][0] / args.steps, 4),
                "track_stats": memo_stats,
                "note": "library default: moments of windows already summed in the same launch are re-used "
                        "(identical results; the headline above re-sums every pass)"}
        ctx.set_track_memo(False)
    h2d = frames_per_step * H * W * 4
    if workload in ("detect", "detect720"):
        d2h = h_rects.numel() * 8 + h_counts.numel() * 4
    elif streams:
        d2h = T * h_events.numel()
    else:
        d2h = h_rects.numel() * 8 + (h_counts.numel() + h_found.numel() + h_objs.numel() + h_wins.numel()) * 4

    # ---- per-rank numbers to rank 0: a scaling loss must be nameable ----
    kernel_ms = {k: round(v[0] / args.steps, 4) for k, v in prof.items()}
    mine = {"rank": rank, "ms_per_step": round(ms_local / args.steps, 4), "kernel_ms_per_step": kernel_ms,
            "gather_ms": None if gather_ms is None else round(gather_ms, 4), "numa": numa,
            "sm_mhz": clocks.get("sm_mhz")}
    per_rank = [mine]
    if world > 1:
        per_rank = [None] * world
        dist.all_gather_object(per_rank, mine)

    if rank == 0:
        peak, peak_src = measured_peaks()
        casc_ms, casc_n = prof["cascade"]
        # SURVEY.md §8(d): one read of the RGBA frame per frame; a k_cascade launch covers one L2 wave of frames
        alg_bytes = frames_per_step * W * H * 4 * args.steps / casc_n if casc_n else None
        achieved = (alg_bytes / 1e9) / (casc_ms / casc_n / 1e3) if casc_n else None
        traffic_pf, traffic_src = captured_traffic(W, H)
        path_gbs = value / world * W * H * 4 / 1e9     # per GPU: the whole path against the HBM-read roofline
        line = {"metric": cfg["metric"], "value": value, "unit": "frames/s",
                "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8+f64",
                "data": "synthetic",
                "config": dict(config_dict(cfg, world, frames_per_step),
                               l2=f"inputs larger than L2 ({frames_per_step * W * H * 4 / 1e6:.0f} MB of frames per GPU per step)"
                                  if frames_per_step * W * H * 4 > 126e6 else "L2 flushed by the step itself: every step streams "
                                  f"{frames_per_step * W * H * 4 / 1e6:.0f} MB of frames and re-writes the pyramid arena",
                               unique_frames=N_UNIQUE if not streams else B * T,
                               track_memo="off (strict: every pass re-summed)",
                               pipeline=("on: the tracking of step s runs on the library's second stream under the detection of "
                                         "step s+1 (ht_set_pipeline); the last step is joined inside the timed region") if pipe
                               else "off (every step completes its own tracking; the pipelined figure is under \"pipelined\")"),
                "e2e": {"value": e2e_value, "unit": "frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "steps": args.steps},
                "gpu_launches": int(launches),
                "roofline": {"bound": "hbm", "kernel": "k_cascade", "achieved": achieved, "peak": peak, "unit": "GB/s",
                             "frac": (achieved / peak) if achieved else None,
                             "traffic": int(traffic_pf * alg_bytes / (W * H * 4)) if (traffic_pf and alg_bytes) else None,
                             "traffic_source": traffic_src,
                             "peak_source": peak_src, "algorithmic_bytes_per_launch": alg_bytes,
                             "kernel_ms_per_launch": casc_ms / casc_n if casc_n else None,
                             "whole_path": {"achieved": path_gbs, "frac": path_gbs / peak,
                                            "note": "value x one RGBA frame read, per GPU (SURVEY 8d's judged fraction)"},
                             "note": "k_cascade is bound by shared-memory load wavefronts and issue slots, not by HBM; "
                                     "see DESIGN.md §5.1 and profiles/"},
                "kernel_ms_per_step": kernel_ms,
                "track_stats": track_stats,
                "per_rank": per_rank,
                "gather": {"ms_per_call": gather_ms, "bytes_per_rank": int(np.prod(rec_shape)) * (4 if rec_dtype == torch.int32 else 1),
                           "overlapped": world > 1,
                           "note": "all_gather_into_tensor of step s runs on its own stream under step s+1"},
                "clocks": clocks}
        if streams:
            ev = d_events.cpu().numpy().view(np.int32).reshape(T, B, 14)
            line["streams"] = {"per_stream_fps": value / (world * B), "offered_fps": 60,
                               "headroom_x": value / (world * B) / 60.0,
                               "frames_in_VJ": int((ev[..., 0] == 1).sum()), "frames_in_CS": int((ev[..., 0] == 2).sum()),
                               "faces_found": int((ev[..., 1] & 1).sum()), "faces_lost": int(((ev[..., 1] >> 1) & 1).sum())}
        if shard_check is not None:
            line["shard_check"] = shard_check
        if other_mode is not None:
            line["unpipelined" if pipe else "pipelined"] = other_mode
        if memo is not None:
            line["memo"] = memo
        if world == 1 and not args.no_cpu_baseline:
            blob = synth.load_cascade_blob()
            if streams:
                cb, _ = cpu_baseline(cfg, min(args.cpu_sample, 16), blob)
            else:
                sample = base if args.cpu_sample <= N_UNIQUE else make_base_frames(W, H, 0, args.cpu_sample)
                oracle_results = []
                cb, _ = cpu_baseline(cfg, args.cpu_sample, blob, frames=sample[: args.cpu_sample], keep=oracle_results)
                # parity of the TIMED batch: frames 0..N_UNIQUE-1 of the batch are the sample frames (roll 0) - what the
                # last timed step left on the device for them must equal what the CPU restatement just computed
                n_chk = min(len(oracle_results), N_UNIQUE, B)
                if workload == "detect_track30" and n_chk:
                    o = last_outputs()
                    got_counts, got_found, got_objs = o[1].cpu().numpy(), o[2].cpu().numpy(), o[3].cpu().numpy()
                    bad = sum(1 for i in range(n_chk)
                              if (int(got_counts[i]), int(got_found[i])) != tuple(oracle_results[i][:2]) or
                              (oracle_results[i][1] and tuple(int(v) for v in got_objs[i, :4]) != tuple(oracle_results[i][2:6])))
                    line["batch_parity"] = {"frames_checked": n_chk, "mismatches": bad,
                                            "what": "detection count, face found, track object x/y/width/height of the last "
                                                    "timed step vs the CPU restatement of the reference on the same frames"}
                    if bad:
                        raise SystemExit(f"bench.py: the timed batch differs from the oracle on {bad} of {n_chk} frames")
                elif workload in ("detect", "detect720") and n_chk:
                    got_counts = d_counts[0].cpu().numpy()
                    bad = sum(1 for i in range(n_chk) if int(got_counts[i]) != oracle_results[i][0])
                    line["batch_parity"] = {"frames_checked": n_chk, "mismatches": bad,
                                            "what": "grouped detection count of the last timed step vs the CPU restatement"}
                    if bad:
                        raise SystemExit(f"bench.py: the timed batch differs from the oracle on {bad} of {n_chk} frames")
            line["cpu_baseline"] = cb
        print(json.dumps(line), flush=True)
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="detect_track30", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=None, help="frames per GPU per step (streams: streams per GPU)")
    ap.add_argument("--streams", type=int, default=None, help="alias of --batch for --workload streams")
    ap.add_argument("--stream-frames", type=int, default=120, help="frames per stream per step (--workload streams)")
    ap.add_argument("--width", type=int, default=None)
    ap.add_argument("--height", type=int, default=None)
    ap.add_argument("--interval", type=int, default=None)
    ap.add_argument("--cpu-sample", type=int, default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--pipeline", type=int, default=int(os.environ.get("HT_BENCH_PIPELINE", "0")),
                    help="detect+track: 0 (default) = every step joins its own tracking, 1 = pipelined steps "
                         "(ht_set_pipeline); on one GPU the other mode is measured too and reported beside the headline")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned as DIR/<name>.npy (float64, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs records the CUDA path (--impl ours)")
    cfg = dict(WORKLOADS[args.workload], workload=args.workload, stream_frames=args.stream_frames)
    for k, v in (("width", args.width), ("height", args.height), ("interval", args.interval),
                 ("batch", args.streams if args.streams is not None else args.batch)):
        if v is not None:
            cfg[k] = v
    if (cfg["width"], cfg["height"]) != (WORKLOADS[args.workload]["width"], WORKLOADS[args.workload]["height"]):
        cfg["metric"] = cfg["metric"].replace(f"{WORKLOADS[args.workload]['width']}x{WORKLOADS[args.workload]['height']}",
                                              f"{cfg['width']}x{cfg['height']}")
    if args.cpu_sample is None:
        # ~10-30 s of CPU work: a 640x480 detect+track frame costs ~0.18 s per core, a 1280x720 detect ~0.45 s
        px = cfg["width"] * cfg["height"] / (640 * 480)
        args.cpu_sample = max(2 * usable_cores(), int(64 / max(px, 0.25))) if args.workload != "streams" else usable_cores()
    if args.impl == "reference":
        run_reference(args, cfg)
    else:
        run_ours(args, cfg)


if __name__ == "__main__":
    main()
