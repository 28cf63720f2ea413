"""Event-fed stream pool slots (TRMStreamPoolOpenEvents): a slot opened with a Monet event list generates its control
frames on the device as it advances, a push giving the number of frames to generate.  Advanced to the end of its list
and flushed, its concatenated output equals TRMBatchSynthesizeEvents of that list with the same voice and settings, bit
for bit (samples, PCM at the utterance's peak, per-push maxima), for any split of the frames over pushes and whatever the
other slots -- event-fed or frame-fed -- do.  An early flush equals the one-shot synthesis of the frames generated so far."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

import oracle_lib as O

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))

gpu = pytest.mark.gpu


def _g():
    import gnuspeech_b200 as g
    return g


def _channels(ip):
    return 2 if ip.channels == 2 else 1


def _peak(mx):
    return mx if mx > 0.0 else 1.0


def _same(got, want, what):
    assert got.shape == want.shape, (what, got.shape, want.shape)
    bad = ~((got == want) | (np.isnan(got) & np.isnan(want)))
    assert np.array_equal(got, want, equal_nan=True), "%s: %d values differ, first at %d" % (
        what, int(bad.sum()), int(np.nonzero(bad)[0][0]))


def _walk(n, nf, seed):
    from gnuspeech_b200 import workloads as W
    return W.random_walk(n, nf, seed=seed).reshape(n, nf, 16)


def _voices(rng, n):
    """male 44.1 kHz, female, a 10 cm tract at 22.05 kHz (down-sampling), stereo at balance 0.3, then random voices."""
    g = _g()
    import fuzz_parity
    female = g.MMSynthesisParameters("Female").inputParameters()
    female.channels = 1
    stereo = g.TRMInputParameters(44100.0, channels=2, balance=0.3)
    vs = [g.TRMInputParameters(44100.0), female, g.TRMInputParameters(22050.0, length=10.0), stereo]
    while len(vs) < n:
        vs.append(fuzz_parity.voice(rng))
    return vs[:n]


def _events_one_shot(ip, ev, fg, prec):
    """TRMBatchSynthesizeEvents of a one-utterance batch -> (samples, interleaved PCM16, maximumSampleValue)."""
    g = _g()
    nf = g.event_list_frame_count(ev)
    b = g.TRMBatch(ip, [nf], precision=prec)
    smp = np.zeros(max(1, b.layout.total_out_samples), b.sample_dtype)
    pcm = np.zeros(max(1, b.layout.total_pcm_samples), np.int16)
    b.synthesize_events(ev, [len(ev)], fg, pcm_out=pcm, samples_out=smp)
    n = int(b.numberSamples[0])
    return smp[:n].copy(), pcm[:n * _channels(ip)].copy(), float(b.maximumSampleValues[0])


def _frames_one_shot(ip, frames, prec):
    """TRMBatch synthesis of whole frames -> (samples, interleaved PCM16, maximumSampleValue)."""
    g = _g()
    b = g.TRMBatch(ip, [frames.shape[0]], precision=prec)
    smp = np.zeros(max(1, b.layout.total_out_samples), b.sample_dtype)
    pcm = np.zeros(max(1, b.layout.total_pcm_samples), np.int16)
    if frames.shape[0]:
        b.synthesize(np.ascontiguousarray(frames), pcm_out=pcm, samples_out=smp, devices=[0])
    n = int(b.numberSamples[0])
    return smp[:n].copy(), pcm[:n * _channels(ip)].copy(), float(b.maximumSampleValues[0])


def _generated(ev, fg):
    """The frames TRMBatchGenerateFrames generates for one list."""
    g = _g()
    b = g.TRMBatch(g.TRMInputParameters(44100.0), [g.event_list_frame_count(ev)], precision=0)
    return b.generate_frames(ev, [len(ev)], fg)[0]


def _cat(parts, dtype):
    return np.concatenate(parts) if parts else np.zeros(0, dtype)


FG_MODES = ["smooth+drift", "plain", "macro only", "per-slot"]


def _fg(mode, k):
    """test_gpu_framegen's generator modes; "per-slot" varies the switches and drift seed per slot k."""
    g = _g()
    if mode == "smooth+drift":
        return g.TRMFrameGeneration()
    if mode == "plain":
        return g.TRMFrameGeneration(useDrift=0, useMacroIntonation=0, useSmoothIntonation=0, useMicroIntonation=1, pitch=-3.5)
    if mode == "macro only":
        return g.TRMFrameGeneration(useDrift=1, useMacroIntonation=1, useSmoothIntonation=0, useMicroIntonation=0,
                                    driftDeviation=0.5, driftCutoff=200.0)
    return g.TRMFrameGeneration(useDrift=(k + 1) % 2, useSmoothIntonation=(k // 2) % 2, useMacroIntonation=1, pitch=-12.0 + k,
                                driftSeed=np.float32(0.1 + 0.17 * k))


def _event_starts(ev):
    """Frame index at which each event after the first becomes current (where a list's interpolation segments meet)."""
    g = _g()
    return [g.event_list_frame_count(ev[:k + 1]) for k in range(1, len(ev))]


@gpu
@pytest.mark.parametrize("precision", [0, 1, 2])
def test_staggered_traffic_event_and_frame_slots(precision):
    """40 requests, half event-fed and half frame-fed, with mixed voices, arrive at different pushes into a pool of 16
    slots (so slots are reused and change kind), advance by random frame counts (0 .. max), are sometimes left out of a
    push and flush at different times."""
    g = _g()
    rng = np.random.default_rng(2000 + precision)
    n_req, cap, mmax = 40, 16, 12
    ips = _voices(rng, n_req)
    is_ev = [k % 2 == 0 for k in range(n_req)]
    evs, fgs, frames, nfs, want = {}, {}, {}, [], []
    for k in range(n_req):
        if is_ev[k]:
            evs[k] = O.synthetic_event_list(3000 + k, float(rng.uniform(0.15, 0.6)), smooth=bool(k % 4 == 0))
            fgs[k] = _fg(FG_MODES[(k // 2) % 4], k)
            nfs.append(g.event_list_frame_count(evs[k]))
            want.append(_events_one_shot(ips[k], evs[k], fgs[k], precision)[0])
        else:
            nfs.append(int(rng.integers(1, 70)))
            frames[k] = _walk(1, nfs[k], seed=3100 + k)[0]
            want.append(_frames_one_shot(ips[k], frames[k], precision)[0])
    start = sorted(int(x) for x in rng.integers(0, 40, n_req))
    pool = g.TRMStreamPool(cap, precision=precision, max_frames_per_push=mmax)
    waiting = list(range(n_req))
    active = {}                                      # slot -> [request, frames sent]
    got = [[] for _ in range(n_req)]
    t = 0
    while waiting or active:
        while waiting and start[waiting[0]] <= t and len(active) < cap:
            k = waiting.pop(0)
            if is_ev[k]:
                s, nf = pool.open_events(ips[k], evs[k], fgs[k])
                assert nf == nfs[k]
            else:
                s = pool.open(ips[k])
            active[s] = [k, 0]
        push, flush = {}, set()
        for s, (k, at) in active.items():
            if rng.random() < 0.2:
                continue                             # not named in this push
            m = min(int(rng.integers(0, mmax + 1)), nfs[k] - at)
            push[s] = m if is_ev[k] else frames[k][at:at + m]
            active[s][1] = at + m
            if at + m == nfs[k] and rng.random() < 0.7:
                flush.add(s)
        out = pool.push(push, flush=flush)
        for s, y in out.items():
            got[active[s][0]].append(y)
        for s in flush:
            del active[s]
        t += 1
    pool.free()
    for k in range(n_req):
        _same(_cat(got[k], want[k].dtype), want[k], "%s request %d" % ("event" if is_ev[k] else "frame", k))


@gpu
@pytest.mark.parametrize("precision", [0, 1, 2])
@pytest.mark.parametrize("mode", FG_MODES)
def test_generator_switches_and_push_patterns(precision, mode):
    """Each generator mode with four push patterns side by side in one pool: one frame per push (every event boundary
    falls on a push boundary), 7 frames (a prime: boundaries inside and at the ends of pushes), the pool's maximum, and
    pushes that end exactly where each event becomes current."""
    g = _g()
    mmax = 40
    ip = g.TRMInputParameters(44100.0)
    smooth = mode in ("smooth+drift", "per-slot")
    evs = [O.synthetic_event_list(4000 + 11 * k, 0.5 + 0.1 * k, smooth=smooth) for k in range(4)]
    fgs = [_fg(mode, k) for k in range(4)]
    nfs = [g.event_list_frame_count(e) for e in evs]
    bounds = _event_starts(evs[3])
    at_bounds = []
    prev = 0
    for b in bounds:
        while b - prev > mmax:
            at_bounds.append(mmax)
            prev += mmax
        at_bounds.append(b - prev)
        prev = b
    patterns = [[1] * nfs[0], [7] * (nfs[1] // 7 + 1), [mmax] * (nfs[2] // mmax + 1), at_bounds]
    pool = g.TRMStreamPool(4, precision=precision, max_frames_per_push=mmax)
    slots = [pool.open_events(ip, evs[k], fgs[k])[0] for k in range(4)]
    got, at, step = [[] for _ in range(4)], [0] * 4, [0] * 4
    live = set(range(4))
    while live:
        push, fl = {}, set()
        for k in list(live):
            m = min(patterns[k][step[k]] if step[k] < len(patterns[k]) else mmax, nfs[k] - at[k])
            step[k] += 1
            push[slots[k]] = m
            at[k] += m
            if at[k] == nfs[k]:
                fl.add(slots[k])
                live.discard(k)
        out = pool.push(push, flush=fl)
        for k in range(4):
            if slots[k] in out:
                got[k].append(out[slots[k]])
    pool.free()
    for k in range(4):
        want = _events_one_shot(ip, evs[k], fgs[k], precision)[0]
        _same(np.concatenate(got[k]), want, "%s, pattern %d" % (mode, k))


@gpu
@pytest.mark.parametrize("precision", [0, 1, 2])
def test_pcm_pushes_reach_the_batch_pcm(precision):
    """PCM pushes of event slots (mono and stereo voices, next to a frame-fed slot) at the utterance's
    maximumSampleValue: the concatenated PCM is TRMBatchSynthesizeEvents' pcm_out and the largest per-push maximum is
    its maximumSampleValue."""
    g = _g()
    rng = np.random.default_rng(50 + precision)
    ips = _voices(rng, 6)
    ips[4] = g.TRMInputParameters(44100.0, channels=2, balance=-1.0)
    evs = [O.synthetic_event_list(5000 + k, 0.4 + 0.1 * k) for k in range(6)]
    fg = g.TRMFrameGeneration()
    want = [_events_one_shot(ips[k], evs[k], fg, precision) for k in range(6)]
    walk = _walk(1, 400, seed=51)[0]
    pool = g.TRMStreamPool(7, precision=precision, max_frames_per_push=16)
    slots = [pool.open_events(ips[k], evs[k])[0] for k in range(6)]
    other = pool.open(ips[5])
    nfs = [g.event_list_frame_count(e) for e in evs]
    pcm, mx, at = [[] for _ in range(6)], [[] for _ in range(6)], [0] * 6
    live = set(range(6))
    t = 0
    while live:
        push, fl = {}, set()
        for k in sorted(live):
            m = min(int(rng.integers(0, 17)), nfs[k] - at[k])
            push[slots[k]] = m
            at[k] += m
            if at[k] == nfs[k]:
                fl.add(slots[k])
                live.discard(k)
        if t % 2:
            push[other] = walk[8 * t:8 * t + 8]
        peak = {slots[k]: _peak(want[k][2]) for k in range(6)}
        peak[other] = 1.0
        out = pool.push_pcm16(push, peak, flush=fl)
        for k in range(6):
            if slots[k] in out:
                pcm[k].append(out[slots[k]][0])
                mx[k].append(out[slots[k]][1])
        t += 1
    pool.free()
    for k in range(6):
        _same(np.concatenate(pcm[k]), want[k][1], "PCM of slot %d (%d channels)" % (k, _channels(ips[k])))
        assert max(mx[k]) == want[k][2], (k, max(mx[k]), want[k][2])


@gpu
def test_different_sample_counts_in_one_cta():
    """Event slots of one voice pushed together with a different frame count each, so that every waveguide CTA holds
    utterances that end after different numbers of blocks (test_gpu_stream_pool's case, with generated frames)."""
    g = _g()
    n, pushes = 20, 6
    ip = g.TRMInputParameters(44100.0)
    evs = [O.synthetic_event_list(6000 + i, 1.0) for i in range(n)]
    nfs = [g.event_list_frame_count(e) for e in evs]
    counts = [[1 + (i * 7 + 3 * k) % n for i in range(n)] for k in range(pushes - 1)]
    counts.append([nfs[i] - sum(c[i] for c in counts) for i in range(n)])
    mmax = max(counts[-1])
    assert min(counts[-1]) > 0
    pool = g.TRMStreamPool(n, precision=0, max_frames_per_push=mmax)
    slots = [pool.open_events(ip, evs[i])[0] for i in range(n)]
    got = [[] for _ in range(n)]
    for k in range(pushes):
        out = pool.push({s: counts[k][i] for i, s in enumerate(slots)}, flush=set(slots) if k == pushes - 1 else ())
        for i, s in enumerate(slots):
            got[i].append(out[s])
    pool.free()
    for i in range(n):
        _same(np.concatenate(got[i]), _events_one_shot(ip, evs[i], g.TRMFrameGeneration(), 0)[0], "slot %d" % i)


@gpu
@pytest.mark.parametrize("precision", [0, 1, 2])
def test_early_flush_and_short_lists(precision):
    """A flush after k of a list's frames equals the one-shot synthesis of the first k frames TRMBatchGenerateFrames
    gives (k = 0, 1, 2 and inside the list); lists of 0 and 1 events expand to no frame, take none, and flush to
    nothing, as the batch gives nothing for them."""
    g = _g()
    N = g._native
    ip = g.TRMInputParameters(44100.0)
    fg = g.TRMFrameGeneration()
    ev = O.synthetic_event_list(7000, 0.8)
    frames = _generated(ev, fg)
    pool = g.TRMStreamPool(6, precision=precision, max_frames_per_push=20)
    for k in (0, 1, 2, 37, frames.shape[0] - 1):
        s, nf = pool.open_events(ip, ev, fg)
        assert nf == frames.shape[0]
        other = pool.open(ip)
        parts, at = [], 0
        walk = _walk(1, 60, seed=k)[0]
        while True:
            m = min(20, k - at)
            last = at + m == k
            out = pool.push({s: m, other: walk[:0]}, flush={s} if last else ())
            parts.append(out[s])
            at += m
            if last:
                break
        pool.close(other)
        _same(_cat(parts, np.float64), _frames_one_shot(ip, frames[:k], precision)[0], "flush after %d frames" % k)
    for n_ev in (0, 1):
        short = ev[:n_ev]
        b = g.TRMBatch(ip, [g.event_list_frame_count(short)], precision=precision)
        assert b.numberSamples[0] == 0
        s, nf = pool.open_events(ip, short, fg)
        assert nf == 0
        with pytest.raises(g.TRMError) as e:
            pool.push({s: 1})
        assert e.value.code == N.TRM_ERR_PARAM
        out = pool.push({s: 0}, flush={s})
        assert out[s].shape == (0,)
    pool.free()


@gpu
@pytest.mark.parametrize("precision", [0, 1, 2])
def test_slot_reuse(precision):
    """One slot event-fed, then frame-fed, then event-fed again (each flushed); another closed in the middle of its list
    and reopened with a new list: every utterance equals its one-shot synthesis."""
    g = _g()
    rng = np.random.default_rng(80 + precision)
    ips = _voices(rng, 5)
    evs = [O.synthetic_event_list(8000 + k, 0.5) for k in range(4)]
    fgs = [_fg("per-slot", k) for k in range(4)]
    walk = _walk(1, 45, seed=81)[0]
    pool = g.TRMStreamPool(2, precision=precision, max_frames_per_push=9)

    def run_events(s, k, ip, flush=True, upto=None):
        nf = g.event_list_frame_count(evs[k]) if upto is None else upto
        parts, at = [], 0
        while at < nf:
            m = min(9, nf - at)
            at += m
            parts.append(pool.push({s: m}, flush={s} if flush and at == nf else ())[s])
        return np.concatenate(parts)

    a, _ = pool.open_events(ips[0], evs[0], fgs[0])
    b, _ = pool.open_events(ips[1], evs[1], fgs[1])
    run_events(b, 1, ips[1], flush=False, upto=30)
    pool.close(b)                                    # client went away in the middle of the list
    b2, _ = pool.open_events(ips[2], evs[2], fgs[2])
    assert b2 == b
    _same(run_events(b2, 2, ips[2]), _events_one_shot(ips[2], evs[2], fgs[2], precision)[0], "reopened after close")
    _same(run_events(a, 0, ips[0]), _events_one_shot(ips[0], evs[0], fgs[0], precision)[0], "event slot")
    a2 = pool.open(ips[3])
    assert a2 == a
    parts = [pool.push({a2: walk[i:i + 9]}, flush={a2} if i + 9 >= 45 else ())[a2] for i in range(0, 45, 9)]
    _same(np.concatenate(parts), _frames_one_shot(ips[3], walk, precision)[0], "frame slot after an event slot")
    a3, _ = pool.open_events(ips[4], evs[3], fgs[3])
    assert a3 == a
    _same(run_events(a3, 3, ips[4]), _events_one_shot(ips[4], evs[3], fgs[3], precision)[0], "event slot after a frame slot")
    pool.free()


@gpu
def test_refusals_leave_the_pool_unchanged():
    """Refused calls change nothing: a push past the end of a list (alone and next to a frame-fed entry) or of more frames
    than the pool takes, a list whose parameter track has no later value (refused by the batch path with the same code),
    a full pool, and a snapshot of an event slot.  After each, the slots continue to their one-shot results."""
    g = _g()
    N = g._native
    ip = g.TRMInputParameters(44100.0)
    down = g.TRMInputParameters(22050.0, length=10.0)
    fg = g.TRMFrameGeneration()
    ev = O.synthetic_event_list(9000, 0.3)
    nf = g.event_list_frame_count(ev)
    walk = _walk(1, 40, seed=91)[0]
    pool = g.TRMStreamPool(3, precision=0, max_frames_per_push=8)
    s, _ = pool.open_events(down, ev, fg)
    f = pool.open(ip)
    got_s, got_f, at_s, at_f = [], [], 0, 0

    def refused(code, fn):
        with pytest.raises(g.TRMError) as e:
            fn()
        assert e.value.code == code

    def step(m_s, m_f, flush=()):
        nonlocal at_s, at_f
        out = pool.push({s: m_s, f: walk[at_f:at_f + m_f]}, flush=flush)
        got_s.append(out[s]); got_f.append(out[f])
        at_s += m_s; at_f += m_f

    step(8, 5)
    bad = ev.copy()
    bad["value"][1:, 4] = np.nan                     # track 4 has no value after the first event
    refused(N.TRM_ERR_PARAM, lambda: pool.open_events(ip, bad, fg))
    b = g.TRMBatch(ip, [g.event_list_frame_count(bad)], precision=0)
    refused(N.TRM_ERR_PARAM, lambda: b.synthesize_events(bad, [len(bad)], fg, pcm_out=np.zeros(max(1, b.layout.total_pcm_samples), np.int16)))
    refused(N.TRM_ERR_PARAM, lambda: pool.push({s: 9, f: walk[at_f:at_f + 3]}))            # more than the pool takes
    refused(N.TRM_ERR_STATE, lambda: pool.save([s]))
    refused(N.TRM_ERR_STATE, lambda: pool.save([f, s]))
    assert len(pool.save([f])[f]) > 0                                                        # frame-fed slots still save
    step(4, 3)
    while at_s + 8 <= nf:
        step(8, 0)
    refused(N.TRM_ERR_PARAM, lambda: pool.push({f: walk[at_f:at_f + 2], s: nf - at_s + 1}))  # past the end of the list
    refused(N.TRM_ERR_PARAM, lambda: pool.push({s: nf - at_s + 1}))
    c, _ = pool.open_events(ip, ev, fg)
    refused(N.TRM_ERR_STATE, lambda: pool.open_events(ip, ev, fg))                           # full
    refused(N.TRM_ERR_STATE, lambda: pool.open(ip))
    pool.close(c)
    step(nf - at_s, 8, flush={s})
    while at_f < 40:
        m = min(8, 40 - at_f)
        out = pool.push({f: walk[at_f:at_f + m]}, flush={f} if at_f + m == 40 else ())
        got_f.append(out[f])
        at_f += m
    pool.free()
    _same(np.concatenate(got_s), _events_one_shot(down, ev, fg, 0)[0], "event slot")
    _same(np.concatenate(got_f), _frames_one_shot(ip, walk, 0)[0], "frame slot")


def test_open_events_needs_a_pool():
    """A NULL pool is refused before anything else (no device needed)."""
    g = _g()
    N = g._native
    ev = O.synthetic_event_list(1, 0.2)
    ip = g.TRMInputParameters(44100.0)
    fg = g.TRMFrameGeneration()
    nf = C.c_int64(-1)
    rc = N.lib().TRMStreamPoolOpenEvents(None, C.byref(ip), ev.ctypes.data_as(C.c_void_p), len(ev), C.byref(fg), C.byref(nf))
    assert rc == N.TRM_ERR_PARAM
    assert nf.value == -1
