"""Time of event-fed stream pool slots (TRMStreamPoolOpenEvents) against frame-fed slots given the same frames, on one GPU.

Workload: n slots (1, 64, 1024) of the default male voice, each with its own 10 s synthetic Monet event list
(tests/oracle_lib.synthetic_event_list), all pushed m frames at a time (m = 5 and 25: 20 and 100 ms).
  events    -- slots opened with the event lists; a push names every slot with m frames to generate on the device
  frames    -- slots of a second pool fed the same frames, generated beforehand with TRMBatchGenerateFrames and
               uploaded by each push
The two pools are pushed alternately in the same run; each time is the median over --reps pushes per pool (after
--warmup pushes each), taken with a host clock around the C call (each push ends in a stream synchronize).
Bytes uploaded per push are counted from shapes: frame-fed, the frames (n * m * 128 B); event-fed, one generator entry
(40 B) and at most two frame-move segments (2 * 24 B) per slot.  The per-push tables both kinds share are not counted.
open -- one slot opened with a 10 s list and closed again, against TRMBatchGenerateFrames of that list (frames copied
to the host, as a frame-fed server needs them); medians over --reps calls after one warm-up call.
The GPU name and power limit are printed first, from the same run.
usage: python tools/stream_pool_events_time.py [--reps 50] [--warmup 5] [--precision 0]"""
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
import oracle_lib as O  # noqa: E402
from gnuspeech_b200 import _native as N  # noqa: E402


def vp(a):
    return a.ctypes.data_as(C.c_void_p)


def timed(fn):
    t0 = time.perf_counter()
    fn()
    return 1e3 * (time.perf_counter() - t0)


def run(prec, n, m, evs, frames, reps, warmup):
    L = N.lib()
    ip = g.TRMInputParameters(44100.0)
    pe = g.TRMStreamPool(n, precision=prec, max_frames_per_push=m)
    pf = g.TRMStreamPool(n, precision=prec, max_frames_per_push=m)
    se = np.array([pe.open_events(ip, evs[i])[0] for i in range(n)], np.int32)
    sf = np.array([pf.open(ip) for _ in range(n)], np.int32)
    cap = max(pe.slot_capacity(), pf.slot_capacity())
    out = np.zeros(n * cap, np.float64 if prec != 1 else np.float32)
    off = np.zeros(n + 1, np.int64)
    nfa = np.full(n, m, np.int32)
    te, tf = [], []
    for k in range(warmup + reps):
        fr = np.ascontiguousarray(frames[:n, k * m:(k + 1) * m])
        a = timed(lambda: N.check(L.TRMStreamPoolPush(pe._h, n, vp(se), vp(nfa), None, None, vp(out), vp(off)), "event push"))
        b = timed(lambda: N.check(L.TRMStreamPoolPush(pf._h, n, vp(sf), vp(nfa), vp(fr), None, vp(out), vp(off)), "frame push"))
        if k >= warmup:
            te.append(a)
            tf.append(b)
    pe.free()
    pf.free()
    return float(np.median(te)), float(np.median(tf))


def open_latency(prec, ev, reps):
    ip = g.TRMInputParameters(44100.0)
    pool = g.TRMStreamPool(1, precision=prec, max_frames_per_push=25)
    b = g.TRMBatch(ip, [g.event_list_frame_count(ev)], precision=prec)
    fg = g.TRMFrameGeneration()

    def open_close():
        s, _ = pool.open_events(ip, ev, fg)
        pool.close(s)
    to, tg = [], []
    for k in range(1 + reps):
        a = timed(open_close)
        c = timed(lambda: b.generate_frames(ev, [len(ev)], fg))
        if k:
            to.append(a)
            tg.append(c)
    pool.free()
    return float(np.median(to)), float(np.median(tg))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--precision", type=int, default=0)
    ap.add_argument("--slots", type=int, nargs="+", default=[1, 64, 1024])
    args = ap.parse_args()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True)
    print("GPU:", q.stdout.strip().splitlines()[0], flush=True)
    n_max = max(args.slots)
    evs = [O.synthetic_event_list(100 + i, 10.0) for i in range(n_max)]
    nfs = [g.event_list_frame_count(e) for e in evs]
    need = (args.warmup + args.reps) * 25
    assert min(nfs) >= need, (min(nfs), need)
    b = g.TRMBatch(g.TRMInputParameters(44100.0), nfs, precision=0)
    allf, _ = b.generate_frames(np.concatenate(evs), [len(e) for e in evs], g.TRMFrameGeneration())
    at = np.concatenate(([0], np.cumsum(nfs)))
    frames = np.stack([allf[at[i]:at[i] + need] for i in range(n_max)])
    ev_bytes = np.mean([e.nbytes for e in evs])
    print("precision %d; 10 s lists: %.0f events, %.1f kB of events, %.0f frames (%.1f kB) on average" % (
        args.precision, np.mean([len(e) for e in evs]), ev_bytes / 1e3, np.mean(nfs), 128 * np.mean(nfs) / 1e3))
    print("%6s %4s %14s %14s %8s %16s %16s" % ("slots", "m", "events ms", "frames ms", "ratio", "events up B", "frames up B"))
    for n in args.slots:
        for m in (5, 25):
            te, tf = run(args.precision, n, m, evs, frames, args.reps, args.warmup)
            print("%6d %4d %14.3f %14.3f %8.2f %16d %16d" % (n, m, te, tf, te / tf, n * (40 + 2 * 24), n * m * 128), flush=True)
    to, tg = open_latency(args.precision, evs[0], args.reps)
    print("open: open_events + close of one 10 s list %.3f ms; TRMBatchGenerateFrames of it (frames to host) %.3f ms" % (to, tg))


if __name__ == "__main__":
    main()
