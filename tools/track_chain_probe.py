#!/usr/bin/env python
"""Probe of k_track's latency chain: kernel time for batches of one repeated frame (heavy / median stream)
at every cluster size.  Usage (GPU box): python tools/track_chain_probe.py"""
import os
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
from headtrackr_b200 import synth  # noqa: E402
from headtrackr_b200.context import Context  # noqa: E402

W, H = 640, 480


def run(frames_np, n_calls=30, reps=3):
    n = frames_np.shape[0]
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx = Context(max_width=W, max_height=H, max_frames=n, device=0, stream=stream.cuda_stream)
    d = torch.from_numpy(frames_np).cuda()
    K = ctx.K
    outs = (torch.zeros(n * K * 12, dtype=torch.int32, device="cuda"), torch.zeros(n, dtype=torch.int32, device="cuda"),
            torch.zeros(n, dtype=torch.int32, device="cuda"), torch.zeros(n * 6, dtype=torch.int32, device="cuda"),
            torch.zeros(n * 4, dtype=torch.int32, device="cuda"))
    ctx.detect_track(d, n_calls=n_calls, outputs=outs)
    torch.cuda.synchronize()
    ctx.profile(True)
    for _ in range(reps):
        ctx.detect_track(d, n_calls=n_calls, outputs=outs)
    torch.cuda.synchronize()
    p = ctx.profile_read()
    st = ctx.debug_track_stats() if hasattr(ctx, "debug_track_stats") else None
    del ctx
    return p["track"][0] / reps, st


def main():
    ids = [int(a) for a in sys.argv[1:]] or [58, 5, 20]
    for fid in ids:
        f = synth.frame(fid, W, H)
        for n in (1, 16):
            batch = np.stack([f] * n)
            for c in (2, 4, 8):
                os.environ["HT_TRACK_CLUSTER"] = str(c)
                ms, st = run(batch)
                print(f"frame {fid} n={n} cluster={c}: track {ms:.3f} ms  stats={st}", flush=True)
    os.environ.pop("HT_TRACK_CLUSTER", None)
    # the bench mix
    frames = np.stack([synth.frame(i, W, H) for i in range(64)])
    for n in (64, 256, 1024):
        batch = np.concatenate([frames] * (n // 64))
        for c in (2, 4):
            os.environ["HT_TRACK_CLUSTER"] = str(c)
            ms, st = run(batch, reps=2)
            print(f"mix n={n} cluster={c}: track {ms:.3f} ms", flush=True)


if __name__ == "__main__":
    main()
