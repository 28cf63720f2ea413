"""Time of stream pool snapshots (TRMStreamPoolSave / TRMStreamPoolRestore) on one GPU, in all three modes.

A pool of 4096 slots of the default male voice is brought into steady traffic (every slot pushed with 100 ms = 25
frames a few times, so each slot carries state, kept history and pending frames).  Then, per mode:
  save n     -- TRMStreamPoolSave of n slots (1, 64, 4096) into a host buffer, blocking
  restore n  -- TRMStreamPoolRestore of those n snapshots into a second pool of 4096 slots (closed again, untimed)
  bytes/slot -- snapshot size of one slot
  push       -- one push of 100 ms to all 4096 slots of the first pool, for scale
Each time is the median of --reps calls after one warm-up call, taken with a host clock around the C call (each call ends
in a stream synchronize).  The GPU name and power limit are printed first, from the same run.
--events times event-fed slots instead: each slot opened with its own 10 s synthetic event list
(tests/oracle_lib.synthetic_event_list) and pushed 25 generated frames a few times; save is TRMStreamPoolSaveAny
(format version 2: the list and the generator state travel with the slot), restore TRMStreamPoolRestore.
usage: python tools/stream_pool_snapshot_time.py [--reps 10] [--slots 4096] [--events]"""
import argparse
import ctypes as C
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import gnuspeech_b200 as g  # noqa: E402
from gnuspeech_b200 import _native as N  # noqa: E402
from gnuspeech_b200 import workloads as W  # noqa: E402


def vp(a):
    return a.ctypes.data_as(C.c_void_p)


def median_ms(fn, reps, after=None):
    fn()
    if after:
        after()
    t = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        t.append(time.perf_counter() - t0)
        if after:
            after()
    return 1e3 * float(np.median(t))


def run(prec, n_slots, reps, frames, events=None):
    """events: one list per slot (event-fed slots, saved with SaveAny), or None (frame-fed slots fed from `frames`)"""
    L = N.lib()
    ip = g.TRMInputParameters(44100.0)
    m = 25
    a = g.TRMStreamPool(n_slots, precision=prec, max_frames_per_push=m + 1)
    b = g.TRMStreamPool(n_slots, precision=prec, max_frames_per_push=m + 1)
    if events is None:
        slots = np.array([a.open(ip) for _ in range(n_slots)], np.int32)
    else:
        slots = np.array([a.open_events(ip, events[i])[0] for i in range(n_slots)], np.int32)
    save = L.TRMStreamPoolSave if events is None else L.TRMStreamPoolSaveAny
    cap = a.slot_capacity()
    out = np.zeros(n_slots * cap, np.float64 if prec != 1 else np.float32)
    off = np.zeros(n_slots + 1, np.int64)
    fl = np.zeros(n_slots, np.uint8)
    pos = [0]

    def push():
        k = pos[0]
        a_, b_ = (0, m + 1) if k == 0 else (1 + k * m, 1 + (k + 1) * m)
        fr = None if events is not None else np.ascontiguousarray(frames[:n_slots, a_:b_])
        N.check(L.TRMStreamPoolPush(a._h, n_slots, vp(slots), vp(np.full(n_slots, b_ - a_, np.int32)),
                                    None if fr is None else vp(fr), vp(fl), vp(out), vp(off)), "push")
        pos[0] += 1

    for _ in range(3):
        push()
    t_push = median_ms(push, reps)
    rows = []
    for n in (1, 64, n_slots):
        sl = np.ascontiguousarray(slots[:n])
        so = np.zeros(n + 1, np.int64)
        N.check(save(a._h, n, vp(sl), None, 0, vp(so)), "size")
        blob = np.zeros(int(so[-1]), np.uint8)
        t_save = median_ms(lambda: N.check(save(a._h, n, vp(sl), vp(blob), blob.size, vp(so)), "save"), reps)
        got = np.zeros(n, np.int32)

        def close_all():
            for s in got:
                b.close(int(s))
        t_restore = median_ms(lambda: N.check(L.TRMStreamPoolRestore(b._h, n, vp(blob), vp(so), vp(got)), "restore"), reps,
                              after=close_all)
        rows.append((n, t_save, t_restore, int(so[-1]) / n))
    a.free()
    b.free()
    return t_push, rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--slots", type=int, default=4096)
    ap.add_argument("--events", action="store_true", help="event-fed slots with 10 s lists, saved with SaveAny")
    args = ap.parse_args()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True)
    print("GPU:", q.stdout.strip().splitlines()[0], flush=True)
    n_pushes = 4 + args.reps
    frames, events = None, None
    if args.events:
        import oracle_lib as O
        events = [O.synthetic_event_list(100 + i, 10.0) for i in range(args.slots)]
        assert min(g.event_list_frame_count(e) for e in events) > 1 + 25 * (n_pushes + 1)
        print("event lists: %.1f events, %.1f kB on average" % (np.mean([len(e) for e in events]),
                                                               np.mean([e.nbytes for e in events]) / 1e3))
    else:
        frames = W.random_walk(args.slots, 1 + 25 * (n_pushes + 1), seed=3).reshape(args.slots, -1, 16)
    print("%-10s %8s %12s %12s %12s %16s" % ("mode", "slots", "save ms", "restore ms", "bytes/slot", "push 100 ms (ms)"))
    for prec, name in ((0, "fp64"), (1, "fp32"), (2, "fp64 strict")):
        t_push, rows = run(prec, args.slots, args.reps, frames, events)
        for n, ts, tr, bps in rows:
            print("%-10s %8d %12.3f %12.3f %12.0f %16s" % (name, n, ts, tr, bps, "%.3f" % t_push if n == args.slots else ""),
                  flush=True)


if __name__ == "__main__":
    main()
