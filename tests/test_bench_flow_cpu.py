"""CPU: bench.py's orchestration (run_ours) executed end to end against a FAKE device layer.

No kernel runs here.  torch.cuda's streams / events and headtrackr_b200.Context are replaced by stand-ins that keep
bench.py's control flow intact, NCCL by gloo; the fake "detector" derives every result record from a checksum of its
input frame.  What this pins, for world 1 and 2, unpipelined and pipelined:
  * every rank issues the same sequence of collectives (a mismatch hangs gloo exactly as it hangs NCCL) - including the
    extra warm-up loop whose exit is decided on rank 0 (the ranks' clocks are skewed on purpose);
  * the lagged, double-buffered result gather delivers the records of the right step (bench.py's own shard_check compares
    what rank 0 received with what it computes for the other rank's frames);
  * the JSON line carries the contract's keys in both modes.
"""
import contextlib
import io
import json
import os
import socket
import sys
import time
from pathlib import Path

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = Path(__file__).resolve().parent.parent


class FakeEvent:
    def __init__(self, enable_timing=False):
        self.t = None

    def record(self, stream=None):
        self.t = time.perf_counter()

    def elapsed_time(self, other):
        return max(1e-3, (other.t - self.t) * 1e3)


class FakeStream:
    cuda_stream = 0

    def __init__(self, priority=0):
        pass

    def wait_event(self, e):
        pass


def checksum(frame):
    return int(np.asarray(frame, dtype=np.int64).sum() % 9973)


class FakeLib:
    """the ctypes entry points the e2e leg calls directly"""

    def __getattr__(self, name):
        return lambda *a, **k: 0


class FakeContext:
    K = 4
    frames_seen = {}

    def __init__(self, max_width, max_height, max_frames, device=0, stream=None, **kw):
        self.launch_count = 0
        self.pipeline = False
        self.pending = None            # (outputs, records) of a pipelined call whose tracking has not been "joined"
        self._L = FakeLib()
        self._h = None

    def _check(self, rc):
        assert rc == 0

    # -- configuration
    def set_track_memo(self, on): pass
    def set_pipeline(self, on):
        self.join()
        self.pipeline = bool(on)
    def stream_reset(self, first=0, n=None): pass
    def profile(self, on): pass
    def profile_read(self, reset=False):
        return {k: (1.0, 1) for k in ("gray", "pyramid", "cascade", "group", "hist", "track_init", "track")}
    def debug_track_stats(self, reset=True):
        return dict(passes=1, serial_passes=0, pixels=1, calls=1, memo_hits=0)
    def close(self): pass

    def join(self):
        if self.pending is not None:
            outs, objs = self.pending
            outs[3][:, 0] = objs          # the deferred "tracking" writes its records only now
            self.pending = None

    # -- work
    def _records(self, frames):
        return torch.tensor([checksum(f) for f in frames.numpy()], dtype=torch.int32)

    def detect_raw(self, frames, interval, mn, out_rects=None, out_counts=None):
        self.launch_count += 1
        if out_counts is None:
            return None, [int(v) for v in self._records(frames)]
        out_counts[:] = self._records(frames)

    def stream_step(self, frames, interval, mn, calc_angles=False, out_events=None):
        self.launch_count += 1

    def detect_track(self, frames, interval, mn, calc_angles=False, n_calls=1, outputs=None):
        self.launch_count += 1
        if not torch.is_tensor(frames):
            frames = torch.from_numpy(np.asarray(frames))
        rec = self._records(frames)
        if outputs is None:
            self.join()
            objs = [dict(x=int(v), y=0, width=0, height=0, angle=0.0) for v in rec]
            return [[] for _ in rec], [1] * len(rec), objs, [(0, 0, 0, 0)] * len(rec)
        if self.pipeline:
            self.join()                 # the previous call's tracking completes before this call's results are due
            outputs[3][:, 0] = -1       # ... while THIS call's records are not there yet
            self.pending = (outputs, rec)
        else:
            outputs[3][:, 0] = rec


def install_fakes():
    torch.cuda.is_available = lambda: True
    torch.cuda.set_device = lambda *_a, **_k: None
    torch.cuda.Stream = FakeStream
    torch.cuda.Event = FakeEvent
    torch.cuda.set_stream = lambda s: None
    torch.cuda.stream = lambda s: contextlib.nullcontext()
    torch.cuda.synchronize = lambda *a, **k: None
    torch.Tensor.cuda = lambda self, *a, **k: self
    for name in ("zeros", "empty", "tensor", "full"):
        real = getattr(torch, name)

        def wrapped(*a, _real=real, **k):
            k.pop("pin_memory", None)
            if k.get("device") in ("cuda",):
                k.pop("device")
            return _real(*a, **k)
        setattr(torch, name, wrapped)
    real_init = dist.init_process_group

    def init(backend, device_id=None, timeout=None, **k):
        return real_init("gloo", **k)
    dist.init_process_group = init

    def all_gather_into_tensor(out, inp, **k):      # gloo's version only takes the concatenated form; NCCL also the stacked one
        parts = [torch.empty_like(inp) for _ in range(out.shape[0])]
        dist.all_gather(parts, inp, **k)
        for r, p in enumerate(parts):
            out[r].copy_(p)
    dist.all_gather_into_tensor = all_gather_into_tensor
    import headtrackr_b200
    headtrackr_b200.Context = FakeContext


def run_bench(rank, world, port, argv, q, skew):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), LOCAL_RANK=str(rank), WORLD_SIZE=str(world))
    sys.path.insert(0, str(ROOT))
    install_fakes()
    if skew:
        time.sleep(skew * rank)         # the ranks reach the warm-up loop at different times: their clocks disagree
    import bench
    bench.ClockSampler.start = lambda self: None
    sys.argv = ["bench.py"] + argv
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        bench.main()
    q.put((rank, buf.getvalue()))


def launch(world, argv, skew=0.0):
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=run_bench, args=(r, world, port, argv, q, skew)) for r in range(world)]
    for p in procs:
        p.start()
    try:
        outs = dict(q.get(timeout=120) for _ in range(world))     # (a hang - mismatched collectives - ends here)
        for p in procs:
            p.join(timeout=60)
            assert p.exitcode == 0
    finally:
        for p in procs:
            if p.is_alive():
                p.terminate()
    return outs


SMALL = ["--width", "64", "--height", "48", "--batch", "8", "--steps", "3", "--warmup", "3", "--no-cpu-baseline"]


@pytest.mark.parametrize("pipeline", [0, 1])
def test_single_rank_line(pipeline):
    out = launch(1, SMALL + ["--pipeline", str(pipeline)])[0]
    line = json.loads(out.strip().splitlines()[-1])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches", "roofline", "clocks"):
        assert key in line, key
    assert line["n_gpus"] == 1 and line["steps"] == 3 and line["value"] > 0
    assert line["gpu_launches"] == 3                                # the fake launches once per step: 3 timed steps
    other = "unpipelined" if pipeline else "pipelined"
    assert other in line and "error" not in line[other] and line[other]["value"] > 0
    assert line["config"]["pipeline"].startswith("on" if pipeline else "off")


@pytest.mark.parametrize("pipeline", [0, 1])
def test_dump_outputs_hold_the_last_timed_step(pipeline, tmp_path):
    """--dump-outputs: the records of the last timed step (pipelined: once its tracking has been joined, not the -1
    placeholders of a step still in flight), as float64, identical on a second run."""
    sys.path.insert(0, str(ROOT))
    import bench
    base = bench.make_base_frames(64, 48, 0, bench.N_UNIQUE)
    want = [checksum(np.roll(base[j % bench.N_UNIQUE], (j // bench.N_UNIQUE) * 16, axis=1)) for j in range(8)]
    dirs = [tmp_path / "a", tmp_path / "b"]
    for d in dirs:
        launch(1, SMALL + ["--pipeline", str(pipeline), "--dump-outputs", str(d)])
    names = sorted(p.name for p in dirs[0].iterdir())
    assert names == ["counts.npy", "found.npy", "frame_index.npy", "objs.npy", "rects.npy", "windows.npy"]
    got = {n: np.load(dirs[0] / n) for n in names}
    assert all(a.dtype == np.float64 and len(a) == 8 for a in got.values())
    assert got["frame_index.npy"].tolist() == list(range(8))
    assert got["objs.npy"].shape == (8, 5) and got["objs.npy"][:, 0].tolist() == want
    assert got["rects.npy"].shape == (8, FakeContext.K, 6)
    for n in names:
        assert np.array_equal(got[n], np.load(dirs[1] / n)), n


@pytest.mark.parametrize("pipeline,workload", [(0, "detect_track30"), (1, "detect_track30"), (0, "detect")])
def test_two_ranks_same_collectives_and_right_records(pipeline, workload):
    """Skewed ranks: a rank-local loop exit or a mis-ordered gather would hang gloo (the queue read times out) or trip
    bench.py's shard_check (rank 0 exits non-zero)."""
    outs = launch(2, SMALL + ["--gpus", "2", "--pipeline", str(pipeline), "--workload", workload], skew=0.15)
    assert outs[1].strip() == ""                                   # only rank 0 prints
    line = json.loads(outs[0].strip().splitlines()[-1])
    assert line["n_gpus"] == 2 and line["value"] > 0
    assert line["shard_check"] == {"ranks_checked": 1, "frames_per_rank": 8, "mismatches": 0}
    assert len(line["per_rank"]) == 2 and line["gather"]["overlapped"] is True


def test_two_ranks_streams_workload(tmp_path):
    """config 5's loop (one ht_stream_step per video frame, T frames per step) on two skewed ranks; --dump-outputs
    holds rank 0's event records of the last step, stream-major."""
    argv = ["--width", "64", "--height", "48", "--streams", "2", "--stream-frames", "4", "--steps", "2", "--warmup", "3",
            "--no-cpu-baseline", "--gpus", "2", "--workload", "streams", "--dump-outputs", str(tmp_path)]
    outs = launch(2, argv, skew=0.15)
    line = json.loads(outs[0].strip().splitlines()[-1])
    assert line["n_gpus"] == 2 and line["value"] > 0 and "streams" in line
    assert sorted(p.name for p in tmp_path.iterdir()) == ["events.npy", "frame_index.npy"]
    ev = np.load(tmp_path / "events.npy")
    assert ev.dtype == np.float64 and ev.shape == (2, 4, 8)
