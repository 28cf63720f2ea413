"""Time of stream pool voice changes (TRMStreamPoolSetVoice) on one GPU, FP64 conformance and FP32 modes.

Pools of 64, 1024 and 4096 slots of the default male voice, pushed with 100 ms (25 frames) per slot until every slot
carries state.  Then, per pool and mode, for n = 1, 64 and all slots, --reps rounds of:
  push        -- an ordinary push of 100 ms to every slot
  set_voice n -- TRMStreamPoolSetVoice of n slots, alternating between two voices with different glottal pulses,
                 breathiness, losses and throat (host describe() of each voice, one upload of the n table rows, one
                 scatter kernel, a stream synchronize)
  push after  -- the push that follows the change, to every slot
Each time is the median over the rounds, taken with a host clock around the C call (every call ends in a stream
synchronize), after one untimed round.  The frames of every push are the same 25 rows per slot: the audio is not the
point here, the work per push is.  The GPU name and power limit are printed first, from the same run.
usage: python tools/stream_pool_voice_time.py [--reps 10] [--pools 64,1024,4096]"""
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

M = 25      # frames per push: 100 ms at 250 Hz


def vp(a):
    return a.ctypes.data_as(C.c_void_p)


def timed(fn):
    t0 = time.perf_counter()
    fn()
    return 1e3 * (time.perf_counter() - t0)


def run(prec, n_slots, reps):
    L = N.lib()
    v1 = g.TRMInputParameters(44100.0)
    v2 = g.TRMInputParameters(44100.0, tp=30.0, tnMin=12.0, tnMax=36.0, breathiness=4.0, lossFactor=1.5, throatVol=12.0)
    pool = g.TRMStreamPool(n_slots, precision=prec, max_frames_per_push=M + 1)
    slots = np.array([pool.open(v1) for _ in range(n_slots)], np.int32)
    frames = np.ascontiguousarray(W.random_walk(n_slots, M, seed=5).reshape(n_slots, M, 16))
    nf = np.full(n_slots, M, np.int32)
    fl = np.zeros(n_slots, np.uint8)
    out = np.zeros(n_slots * pool.slot_capacity(), np.float64 if prec != 1 else np.float32)
    off = np.zeros(n_slots + 1, np.int64)

    def push():
        N.check(L.TRMStreamPoolPush(pool._h, n_slots, vp(slots), vp(nf), vp(frames), vp(fl), vp(out), vp(off)), "push")

    voices = {}
    for v in (v1, v2):
        arr = (N.TRMInputParametersStruct * n_slots)()
        for i in range(n_slots):
            C.memmove(C.byref(arr[i]), C.byref(v), C.sizeof(v))
        voices[id(v)] = arr
    ts = np.zeros(n_slots, np.int64)
    os_ = np.zeros(n_slots, np.int64)

    def set_voice(n, v):
        N.check(L.TRMStreamPoolSetVoice(pool._h, n, vp(slots), voices[id(v)], vp(ts), vp(os_)), "set_voice")

    for _ in range(3):
        push()
    rows = []
    for n in sorted({1, 64, n_slots}):
        t_push, t_set, t_after = [], [], []
        for r in range(reps + 1):
            v = v2 if r % 2 == 0 else v1
            a, b, c = timed(push), timed(lambda: set_voice(n, v)), timed(push)
            if r:
                t_push.append(a)
                t_set.append(b)
                t_after.append(c)
        set_voice(n_slots, v1)
        rows.append((n, float(np.median(t_push)), float(np.median(t_set)), float(np.median(t_after))))
    pool.free()
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--pools", default="64,1024,4096")
    args = ap.parse_args()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True)
    print("GPU:", q.stdout.strip().splitlines()[0], flush=True)
    print("%-6s %6s %8s %10s %14s %14s" % ("mode", "pool", "changed", "push ms", "set_voice ms", "push after ms"))
    for prec, name in ((0, "fp64"), (1, "fp32")):
        for n_slots in [int(x) for x in args.pools.split(",")]:
            for n, tp, tv, ta in run(prec, n_slots, args.reps):
                print("%-6s %6d %8d %10.3f %14.3f %14.3f" % (name, n_slots, n, tp, tv, ta), flush=True)


if __name__ == "__main__":
    main()
