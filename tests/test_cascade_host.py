"""CPU: k_cascade's tile evaluation emulated on the host with the kernel's own ingredients.

ht_api.cu, built with -DHT_HOST_SELFTEST, compiles for the CPU the SAME generated stage code
(cascade_face_gen.inc: quad-form truth tables, byte-form integer sums), the same tile layout (`point_word`, parity-
split level 0, interleaved level-2 copies), the same staging index arithmetic, the same late-stage schedule and
integer thresholds as k_cascade, and replaces only the parallel execution by loops.  Fed with a frame-quad-
interleaved arena built from the oracle's pyramid planes, its raw detection lists must equal the oracle's
(src/ccv.js:178-243) bit for bit.  This pins on the CPU everything of the kernel that is arithmetic or layout; what
remains for the GPU tests is the CUDA plumbing (staging copies, lists, barriers) and the pyramid kernels.
"""
import ctypes as C
import subprocess
from pathlib import Path

import numpy as np
import pytest

import oracle
from headtrackr_b200 import synth

ROOT = Path(__file__).resolve().parent.parent
CSRC = ROOT / "headtrackr_b200" / "csrc"


@pytest.fixture(scope="module")
def st(tmp_path_factory):
    so = tmp_path_factory.mktemp("selftest") / "libht_selftest.so"
    subprocess.check_call(["/usr/local/cuda/bin/nvcc", "-DHT_HOST_SELFTEST", "-gencode", "arch=compute_100a,code=sm_100a",
                           "-O2", "-std=c++17", "-fmad=false", "-Xcompiler", "-fPIC", "-shared", "-o", str(so),
                           str(CSRC / "ht_api.cu")], stderr=subprocess.DEVNULL)
    L = C.CDLL(str(so))
    L.ht_selftest_planes.argtypes = [C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int]
    L.ht_selftest_cascade.argtypes = [C.c_char_p, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int,
                                      C.c_int, C.c_void_p, C.c_void_p, C.c_int]
    return L


def quad_arena(st, frames, W, H, interval):
    """The device layout of one frame quad: one word per pixel, byte f = frame f (planes from the oracle)."""
    info = np.zeros(2 + 6 * 256, np.int32)
    assert st.ht_selftest_planes(W, H, interval, info.ctypes.data, info.size) == 0
    n_planes, stride = int(info[0]), int(info[1])
    arena = np.zeros(stride, np.uint32)
    pyrs = [oracle.Pyramid(oracle.grayscale(f), interval) for f in frames]
    for i in range(n_planes):
        off, pitch, w, h, slot, q = (int(v) for v in info[2 + 6 * i: 8 + 6 * i])
        view = arena[off: off + pitch * h].reshape(h, pitch)
        for f, p in enumerate(pyrs):
            pl = p.plane(slot, q)
            assert pl.shape == (h, w)
            view[:, :w] |= pl.astype(np.uint32) << (8 * f)
    return arena


def run(st, blob, frames, W, H, interval=5, force_ties=0, quad_stages=2, cap=8192):
    arena = quad_arena(st, frames, W, H, interval)
    out = np.zeros((4, cap, 4), np.float64)
    counts = np.zeros(4, np.int32)
    rc = st.ht_selftest_cascade(blob, len(blob), W, H, interval, arena.ctypes.data, len(frames), force_ties, quad_stages,
                                out.ctypes.data, counts.ctypes.data, cap)
    assert rc == 0
    return [[tuple(out[f, i]) for i in range(counts[f])] for f in range(4)]


def want_raw(frame, blob, interval=5):
    return [(r[0], r[1], r[2], r[4]) for r in oracle.detect(frame, blob, interval, 0)]


@pytest.mark.parametrize("W,H,interval", [(160, 120, 5), (320, 240, 5), (171, 133, 3)])
def test_emulated_tiles_equal_the_oracle(st, blob, W, H, interval):
    frames = [synth.frame(i, W, H) for i in range(3)] + [synth.frame(9, W, H, kind="noise")]
    got = run(st, blob, frames, W, H, interval)
    total = 0
    for f in range(4):
        want = want_raw(frames[f], blob, interval)
        assert got[f] == want, f
        total += len(want)
    assert total >= 3                                       # parity must not be vacuous


def test_partial_quad_and_forced_ties(st, blob):
    W, H = 320, 240
    frames = [synth.frame(40 + i, W, H) for i in range(3)]
    base = run(st, blob, frames, W, H)
    assert base[3] == []
    for f in range(3):
        assert base[f] == want_raw(frames[f], blob) and base[f]
    # every integer / truth-table decision replaced by the reference's ordered fp64 adds: same lists
    assert run(st, blob, frames, W, H, force_ties=3) == base


def test_bench_resolution_frame(st, blob):
    W, H = 640, 480
    frames = [synth.frame(i, W, H) for i in (0, 3)]
    got = run(st, blob, frames, W, H)
    for f in range(2):
        assert got[f] == want_raw(frames[f], blob)
        assert len(got[f]) >= 5
