"""Latency / throughput of the stream pool (TRMStreamPool) against lockstep TRMStream, on one GPU.

Rows: n active slots x pushes of m frames (4 ms each), FP64 and FP32:
  pool     -- n slots of the default male voice, every slot pushed with m frames (the lockstep shape through the pool)
  pool pcm -- the same slots and frames through TRMStreamPoolPushPCM16 (mono PCM16 instead of samples; also for mixed)
  stream   -- the same through one TRMStream of n streams
  mixed    -- n slots at random positions with three voices (male 44.1 kHz, female, 10 cm tract at 22.05 kHz),
              random frame counts 0..m per slot and push, 10 % of the slots flushing or opening per push
Each time is the median of >= 20 pushes after warm-up pushes, taken with a host clock around the C call (a push ends in a
stream synchronize).  The GPU name and power limit are printed first, from the same run.
usage: python tools/stream_pool_time.py [--pushes 20] [--warmup 3]"""
import argparse
import ctypes as C
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import gnuspeech_b200 as g  # noqa: E402
from gnuspeech_b200 import _native as N  # noqa: E402
from gnuspeech_b200 import workloads as W  # noqa: E402


def vp(a):
    return a.ctypes.data_as(C.c_void_p)


class Push(object):
    """One pool push into pageable numpy buffers: samples (TRMStreamPoolPush), or PCM16 scaled against a fixed peak
    with the per-entry maxima (TRMStreamPoolPushPCM16)."""

    def __init__(self, pool, n, prec, pcm):
        self.pool, self.pcm = pool, pcm
        cap = pool.slot_capacity()
        self.off = np.zeros(n + 1, np.int64)
        if pcm:
            self.out = np.zeros(2 * n * cap, np.int16)
            self.peak = np.ones(n, np.float64)
            self.mx = np.zeros(n, np.float64)
        else:
            self.out = np.zeros(n * cap, np.float64 if prec != 1 else np.float32)

    def __call__(self, slots, nf, fr, fl):
        L, h, n = N.lib(), self.pool._h, len(slots)
        if self.pcm:
            N.check(L.TRMStreamPoolPushPCM16(h, n, vp(slots), vp(nf), vp(fr), vp(fl), vp(self.peak), vp(self.out), vp(self.off),
                                             vp(self.mx)), "push pcm16")
        else:
            N.check(L.TRMStreamPoolPush(h, n, vp(slots), vp(nf), vp(fr), vp(fl), vp(self.out), vp(self.off)), "push")


def pool_lockstep(prec, n, m, frames, warm, reps, pcm=False):
    ip = g.TRMInputParameters(44100.0)
    pool = g.TRMStreamPool(n, precision=prec, max_frames_per_push=m + 1)
    slots = np.array([pool.open(ip) for _ in range(n)], np.int32)
    push = Push(pool, n, prec, pcm)
    fl = np.zeros(n, np.uint8)
    t = []
    for k in range(warm + reps):
        a, b = (0, m + 1) if k == 0 else (1 + k * m, 1 + (k + 1) * m)
        fr = np.ascontiguousarray(frames[:n, a:b])
        nf = np.full(n, b - a, np.int32)
        t0 = time.perf_counter()
        push(slots, nf, fr, fl)
        if k >= warm:
            t.append(time.perf_counter() - t0)
    pool.free()
    return float(np.median(t))


def stream_lockstep(prec, n, m, frames, warm, reps):
    ip = g.TRMInputParameters(44100.0)
    st = g.TRMStream(n, ip, precision=prec, max_frames_per_push=m + 1)
    k_out = C.c_int64(0)
    t = []
    for k in range(warm + reps):
        a, b = (0, m + 1) if k == 0 else (1 + k * m, 1 + (k + 1) * m)
        fr = np.ascontiguousarray(frames[:n, a:b])
        t0 = time.perf_counter()
        N.check(N.lib().TRMStreamPush(st._h, vp(fr), b - a, 0, vp(st._buf), C.byref(k_out)), "push")
        if k >= warm:
            t.append(time.perf_counter() - t0)
    st.free()
    return float(np.median(t))


def pool_mixed(prec, n, m, frames, warm, reps, pcm=False, seed=5):
    rng = np.random.default_rng(seed)
    female = g.MMSynthesisParameters("Female").inputParameters()
    female.channels = 1
    voices = [g.TRMInputParameters(44100.0), female, g.TRMInputParameters(22050.0, length=10.0)]
    pool = g.TRMStreamPool(n, precision=prec, max_frames_per_push=m)
    pos = {}                                             # slot -> frames sent (row into `frames`)
    for i in range(n):
        pos[pool.open(voices[i % 3])] = int(rng.integers(0, 40))     # random positions in the frame tracks
    push = Push(pool, n, prec, pcm)
    t, audio = [], []
    # every slot's first push: bring it to its position
    for k in range(warm + reps):
        slots = np.array(sorted(pos), np.int32)
        nf = rng.integers(0, m + 1, len(slots)).astype(np.int32) if k else np.full(len(slots), m, np.int32)
        fl = (rng.random(len(slots)) < 0.05).astype(np.uint8) if k else np.zeros(len(slots), np.uint8)
        rows = [frames[s % frames.shape[0], pos[s]:pos[s] + c] for s, c in zip(slots, nf)]
        nf = np.array([r.shape[0] for r in rows], np.int32)
        fr = np.ascontiguousarray(np.concatenate(rows))
        t0 = time.perf_counter()
        push(slots, nf, fr, fl)
        dt = time.perf_counter() - t0
        if k >= warm:
            t.append(dt)
            audio.append(float(nf.sum()) * 0.004)
        for s, c, f in zip(slots, nf, fl):
            pos[int(s)] += int(c)
            if f or pos[int(s)] + m >= frames.shape[1]:
                if not f:
                    pool.close(int(s))
                del pos[int(s)]
        while len(pos) < n:                              # as many new requests as ended
            pos[pool.open(voices[int(rng.integers(0, 3))])] = 0
    pool.free()
    i = int(np.argsort(t)[len(t) // 2])
    return t[i], audio[i]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pushes", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--sizes", default="1,64,1024,4096")
    args = ap.parse_args()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True)
    print("GPU:", q.stdout.strip().splitlines()[0], flush=True)
    sizes = [int(x) for x in args.sizes.split(",")]
    reps, warm = args.pushes, args.warmup
    m_max = 25
    frames = W.random_walk(max(sizes), 1 + (warm + reps + 1) * m_max, seed=3).reshape(max(sizes), -1, 16)
    print("%-5s %-6s %6s %6s %11s %11s %11s %7s %9s %12s" % ("prec", "shape", "slots", "push", "pool ms", "pool pcm ms",
                                                            "stream ms", "ratio", "pcm/pool", "audio-s/s"), flush=True)
    for prec, name in ((0, "fp64"), (1, "fp32")):
        for n in sizes:
            for m in (5, 25):
                tp = pool_lockstep(prec, n, m, frames, warm, reps)
                tq = pool_lockstep(prec, n, m, frames, warm, reps, pcm=True)
                ts = stream_lockstep(prec, n, m, frames, warm, reps)
                print("%-5s %-6s %6d %4dms %11.3f %11.3f %11.3f %7.2f %9.2f %12.0f" % (
                    name, "lock", n, m * 4, tp * 1e3, tq * 1e3, ts * 1e3, tp / ts, tq / tp, n * m * 0.004 / tp), flush=True)
        for n in sizes[-2:]:
            for m in (5, 25):
                tm, audio = pool_mixed(prec, n, m, frames, warm, reps)
                tq, _ = pool_mixed(prec, n, m, frames, warm, reps, pcm=True)
                print("%-5s %-6s %6d %4dms %11.3f %11.3f %11s %7s %9.2f %12.0f" % (
                    name, "mixed", n, m * 4, tm * 1e3, tq * 1e3, "-", "-", tq / tm, audio / tm), flush=True)


if __name__ == "__main__":
    main()
