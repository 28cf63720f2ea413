"""Snapshots of event-fed stream pool slots (TRMStreamPoolSaveAny, format version 2): the event list and the frame
generator's state travel with the stream.  A restored event slot, advanced to the end of its list and flushed, gives output
that, appended to what the saved slot returned before the save, equals TRMBatchSynthesizeEvents bit for bit (samples, PCM
at the utterance's peak, per-push maxima); an early flush equals the one-shot synthesis of the frames generated so far.
Refused restores leave both pools exactly as they were."""
import ctypes as C
import struct

import numpy as np
import pytest

import oracle_lib as O
from test_gpu_stream_pool_events import FG_MODES, _event_starts, _events_one_shot, _fg, _frames_one_shot, _generated
from test_gpu_stream_pool_snapshot import (AT_COUNTERS, FIXED, Request, _built_snapshot, _counters, _device_count,
                                           _one_shot, _peak, _rate_voice, _reseal, _same, _voices, _walk)

gpu = pytest.mark.gpu

# the version-2 layout include/trm.h documents
EVHEADER, GEN, EVENT = 72, 600, 296
AT_GEN_I = 552                       # i, now, next inside the generator state


def _g():
    import gnuspeech_b200 as g
    return g


def _ev_header(b):
    """(n_events, list_frames, generator flag) of a version-2 snapshot"""
    n_events, list_frames = struct.unpack_from("<qq", b, FIXED)
    return n_events, list_frames, struct.unpack_from("<I", b, FIXED + 64)[0]


def _at_gen(b):
    """byte offset of the generator state of a version-2 snapshot with generator = 1"""
    return len(b) - _ev_header(b)[0] * EVENT - GEN


def _at_list(b):
    return len(b) - _ev_header(b)[0] * EVENT


class EvRequest(Request):
    """Request for an event slot: pushes take frame counts, the wanted result is TRMBatchSynthesizeEvents'."""

    def __init__(self, k, ip, ev, fg, precision, pcm_only=False):
        g = _g()
        self.ev, self.fg, self.nf = ev, fg, g.event_list_frame_count(ev)
        Request.__init__(self, k, ip, None, _events_one_shot(ip, ev, fg, precision), pcm_only)

    def open(self, pool):
        return pool.open_events(self.ip, self.ev, self.fg)[0]

    def take(self, m):
        m = min(m, self.nf - self.sent)
        self.sent += m
        return m


class FrRequest(Request):
    def __init__(self, k, ip, frames, want, pcm_only=False):
        Request.__init__(self, k, ip, frames, want, pcm_only)
        self.nf = frames.shape[0]

    def open(self, pool):
        return pool.open(self.ip)

    def take(self, m):
        m = min(m, self.nf - self.sent)
        self.sent += m
        return self.frames[self.sent - m:self.sent]


def _push(pool, active, rng, mmax, as_pcm, p_skip=0.2):
    """One push of pool: each active request (slot -> request) named with prob. 1 - p_skip, advanced by 0..mmax frames;
    a request at the end of its frames flushes with prob. 0.7.  Checks the outputs."""
    push, flush = {}, set()
    for s, r in active.items():
        if rng.random() < p_skip or (r.pcm_only and not as_pcm):
            continue
        push[s] = r.take(int(rng.integers(0, mmax + 1)))
        if r.sent == r.nf and rng.random() < 0.7:
            flush.add(s)
    if not push and not flush:
        return
    if as_pcm:
        out = pool.push_pcm16(push, {s: _peak(active[s].want[2]) for s in set(push) | flush}, flush=flush)
        for s, (pcm, m) in out.items():
            active[s].got_pcm(pcm, m)
    else:
        for s, y in pool.push(push, flush=flush).items():
            active[s].got_samples(y)
    for s in flush:
        del active[s]


def _migrate(rng, src, src_active, dst, dst_active, p):
    """Moves each slot of src with prob. p through one SaveAny of the mixed set and one Restore, as far as dst has room.
    Returns the requests moved."""
    pick = [s for s in src_active if rng.random() < p][:dst.capacity - len(dst_active)]
    if not pick:
        return []
    snaps = src.save(pick, event_slots=True)
    for s in pick:
        src.close(s)
    moved = []
    for s, n in zip(pick, dst.restore([snaps[s] for s in pick])):
        dst_active[n] = src_active.pop(s)
        moved.append(dst_active[n])
    return moved


def _traffic(precision, dev_b, seed):
    g = _g()
    rng = np.random.default_rng(seed)
    n_req = 36
    ips = _voices(rng, n_req)
    reqs = []
    frame_k = [k for k in range(n_req) if k % 2]
    walks = {k: _walk(1, int(rng.integers(1, 70)), seed=seed * 7 + k)[0] for k in frame_k}
    want = dict(zip(frame_k, _one_shot([ips[k] for k in frame_k], [walks[k] for k in frame_k], precision)))
    for k in range(n_req):
        if k % 2 == 0:
            ev = O.synthetic_event_list(seed * 3 + k, float(rng.uniform(0.1, 0.4)), smooth=bool(k % 4 == 0))
            reqs.append(EvRequest(k, ips[k], ev, _fg(FG_MODES[(k // 2) % 4], k), precision, pcm_only=(k % 3 == 0)))
        else:
            reqs.append(FrRequest(k, ips[k], walks[k], want[k], pcm_only=(k % 3 == 0)))
    start = sorted(int(x) for x in rng.integers(0, 25, n_req))
    a = g.TRMStreamPool(20, precision=precision, max_frames_per_push=12)
    b = g.TRMStreamPool(15, precision=precision, max_frames_per_push=9, device=dev_b)
    a_act, b_act = {}, {}
    waiting = list(range(n_req))
    moved, t = 0, 0
    ev_moved = set()
    while waiting or a_act or b_act:
        while waiting and start[waiting[0]] <= t and len(a_act) < a.capacity:
            r = reqs[waiting.pop(0)]
            a_act[r.open(a)] = r
        _push(a, a_act, rng, a.max_frames_per_push, bool(rng.random() < 0.5))
        _push(b, b_act, rng, b.max_frames_per_push, bool(rng.random() < 0.5))
        for src, sa, dst, da, p in ((a, a_act, b, b_act, 0.15), (b, b_act, a, a_act, 0.08)):
            for r in _migrate(rng, src, sa, dst, da, p):
                moved += 1
                if isinstance(r, EvRequest):
                    ev_moved.add(r.k)
        t += 1
    a.free()
    b.free()
    for r in reqs:
        r.finished()
    assert moved >= 20 and len(ev_moved) >= 6, (moved, len(ev_moved))


@gpu
@pytest.mark.parametrize("precision", [0, 1, 2])
def test_migration_under_staggered_traffic(precision):
    """Event and frame slots with mixed voices move both ways between pools of different capacity and
    max_frames_per_push, one SaveAny per move of a mixed set; float and PCM pushes mix."""
    _traffic(precision, 0, 600 + precision)


@gpu
@pytest.mark.parametrize("precision", [0, 1, 2])
def test_migration_across_devices(precision):
    if _device_count() < 2:
        pytest.skip("one CUDA device: the second pool of the migration test would be on the same device")
    _traffic(precision, 1, 700 + precision)


def _serve(pool, slot, r, rng, mmax, pcm_every=2):
    """Pushes r's remaining frames through slot and flushes; alternates float and PCM pushes."""
    k = 0
    while True:
        fr = {slot: r.take(int(rng.integers(1, mmax + 1)))}
        last = r.sent == r.nf
        if k % pcm_every:
            pcm, mx = pool.push_pcm16(fr, _peak(r.want[2]), flush={slot} if last else ())[slot]
            r.got_pcm(pcm, mx)
        else:
            r.got_samples(pool.push(fr, flush={slot} if last else ())[slot])
        k += 1
        if last:
            return


def _advance(pool, slot, r, upto, mmax):
    while r.sent < upto:
        r.got_samples(pool.push({slot: r.take(min(mmax, upto - r.sent))})[slot])


@gpu
@pytest.mark.parametrize("precision", [0, 1, 2])
def test_save_points(precision):
    """Saved never pushed (no generator part), after 1 frame, inside a control interval, exactly where an event becomes
    current, one frame before the end of the list, at its end before the flush, and at control periods 8 and 19,794;
    restored into a pool whose rows and SlotCapacity must grow, each continues to its one-shot result."""
    g = _g()
    rng = np.random.default_rng(110 + precision)
    male = g.TRMInputParameters(44100.0)
    fg = g.TRMFrameGeneration()
    ev = O.synthetic_event_list(111, 0.5)
    nf = g.event_list_frame_count(ev)
    starts = _event_starts(ev)
    short = O.synthetic_event_list(112, 0.12)
    cases = [("never pushed", male, ev, 0), ("one frame", male, ev, 1), ("mid interval", male, ev, 13),
             ("event start", male, ev, starts[4]), ("one before the end", male, ev, nf - 1), ("end", male, ev, nf),
             ("period 8", _rate_voice(2500.0), ev, 57), ("period 19794", _rate_voice(1.0), short, 3)]
    a = g.TRMStreamPool(len(cases), precision=precision, max_frames_per_push=5)
    reqs, slots = [], []
    for i, (name, ip, e, before) in enumerate(cases):
        r = EvRequest(i, ip, e, fg, precision)
        s = r.open(a)
        _advance(a, s, r, before, 5)
        reqs.append(r)
        slots.append(s)
    snaps = a.save(slots, event_slots=True)
    for (name, ip, e, before), s in zip(cases, slots):
        b = snaps[s]
        assert struct.unpack_from("<I", b, 8)[0] == 2
        assert _ev_header(b) == (len(e), g.event_list_frame_count(e), 1 if before else 0), name
        info = g.snapshot_info(b)["events"]
        assert info["frames_generated"] == before and info["list_frames"] == g.event_list_frame_count(e), name
    assert len(snaps[slots[0]]) == FIXED + EVHEADER + len(ev) * EVENT          # never pushed: no data but the list
    mid = _counters(snaps[slots[2]])
    assert mid[6] == 0 and mid[1] % g.derive(male, 2).controlPeriod != 0
    assert _counters(snaps[slots[7]])[1] % 19794 != 0
    for s in slots:
        a.close(s)
    b = g.TRMStreamPool(len(cases) + 2, precision=precision, max_frames_per_push=2)
    cap0 = b.slot_capacity()
    new = b.restore([snaps[s] for s in slots])
    assert b.slot_capacity() > cap0
    for r, s in zip(reqs, new):
        _serve(b, s, r, rng, 2)
        r.finished()
    a.free()
    b.free()


@gpu
@pytest.mark.parametrize("precision", [0, 1, 2])
@pytest.mark.parametrize("mode", FG_MODES)
def test_generator_modes(precision, mode):
    """Every generator mode, with per-slot drift seeds and smooth intonation: slots saved in the middle of an intonation
    segment (between two event starts) and restored into another pool continue to TRMBatchSynthesizeEvents."""
    g = _g()
    rng = np.random.default_rng(120 + precision)
    smooth = mode in ("smooth+drift", "per-slot")
    ip = g.TRMInputParameters(44100.0)
    evs = [O.synthetic_event_list(121 + 5 * k, 0.4 + 0.1 * k, smooth=smooth) for k in range(4)]
    reqs = [EvRequest(k, ip, evs[k], _fg(mode, k), precision) for k in range(4)]
    a = g.TRMStreamPool(4, precision=precision, max_frames_per_push=16)
    slots = [r.open(a) for r in reqs]
    for k, (r, s) in enumerate(zip(reqs, slots)):
        st = _event_starts(evs[k])
        j = 2 + k
        assert st[j + 1] - st[j] >= 2
        _advance(a, s, r, (st[j] + st[j + 1]) // 2, 16)
    snaps = a.save(slots, event_slots=True)
    a.free()
    b = g.TRMStreamPool(5, precision=precision, max_frames_per_push=7)
    for r, s in zip(reqs, b.restore([snaps[s] for s in slots])):
        _serve(b, s, r, rng, 7)
        r.finished()
    b.free()


@gpu
@pytest.mark.parametrize("precision", [0, 1, 2])
def test_forks(precision):
    """A fork, a fork of a fork and one snapshot restored twice all continue to the one-shot result; an early flush of a
    fork equals the one-shot synthesis of the frames generated so far."""
    g = _g()
    ip = g.TRMInputParameters(22050.0, length=10.0, channels=2, balance=0.3)
    fg = _fg("per-slot", 3)
    ev = O.synthetic_event_list(130, 0.6)
    nf = g.event_list_frame_count(ev)
    want = _events_one_shot(ip, ev, fg, precision)
    pool = g.TRMStreamPool(8, precision=precision, max_frames_per_push=9)
    src = EvRequest(0, ip, ev, fg, precision)
    s0 = src.open(pool)
    _advance(pool, s0, src, 41, 9)
    head = want[0][:src.pos]
    snap = pool.save([s0], event_slots=True)[s0]
    c1, c2 = pool.restore([snap, snap])
    br = {s0: src}
    for s in (c1, c2):
        r = EvRequest(0, ip, ev, fg, precision)
        r.sent, r.pos = src.sent, src.pos
        br[s] = r
    for s, r in br.items():
        _advance(pool, s, r, r.sent + 11, 4)
    c3 = pool.restore([pool.save([c1], event_slots=True)[c1]])[0]          # fork of the fork
    br[c3] = EvRequest(0, ip, ev, fg, precision)
    br[c3].sent, br[c3].pos = br[c1].sent, br[c1].pos
    # early flush of a fork, k frames after the prefix
    c4 = pool.restore([snap])[0]
    k = 41 + 7
    tail = [pool.push({c4: 7}, flush={c4})[c4]]
    frames = _generated(ev, fg)
    _same(np.concatenate([head] + tail), _frames_one_shot(ip, frames[:k], precision)[0], "early flush of a fork")
    rng = np.random.default_rng(131)
    for s, r in br.items():
        _serve(pool, s, r, rng, 9)
        r.finished()
    assert pool.save([], event_slots=True) == {}
    pool.free()
    assert nf > 60


@gpu
@pytest.mark.parametrize("precision", [0, 1, 2])
def test_storage_reuse(precision):
    """A restore into a pool that never opened an event slot; into a slot whose earlier list was longer, then shorter;
    and one slot used as restored event slot, then frame slot, then restored event slot again."""
    g = _g()
    rng = np.random.default_rng(140 + precision)
    ip = g.TRMInputParameters(44100.0)
    fg = g.TRMFrameGeneration()
    long_ev, short_ev = O.synthetic_event_list(141, 0.8), O.synthetic_event_list(142, 0.2)
    src = g.TRMStreamPool(2, precision=precision, max_frames_per_push=6)
    rl, rs = EvRequest(0, ip, long_ev, fg, precision), EvRequest(1, ip, short_ev, fg, precision)
    sl, ss = rl.open(src), rs.open(src)
    _advance(src, sl, rl, 20, 6)
    _advance(src, ss, rs, 9, 6)
    snaps = src.save([sl, ss], event_slots=True)
    src.free()

    def copy(r):
        c = EvRequest(r.k, r.ip, r.ev, r.fg, precision)
        c.sent, c.pos = r.sent, r.pos
        return c

    dst = g.TRMStreamPool(1, precision=precision, max_frames_per_push=5)      # never opened an event slot
    s = dst.restore([snaps[ss]])[0]
    r = copy(rs)
    _serve(dst, s, r, rng, 5)
    r.finished()
    s = dst.restore([snaps[sl]])[0]                                          # the slot's list storage grows
    r = copy(rl)
    _serve(dst, s, r, rng, 5)
    r.finished()
    s = dst.restore([snaps[ss]])[0]                                          # a shorter list in the longer storage
    r = copy(rs)
    _serve(dst, s, r, rng, 5)
    r.finished()
    walk = _walk(1, 33, seed=143)[0]
    fr = FrRequest(2, ip, walk, _frames_one_shot(ip, walk, precision))
    _serve(dst, fr.open(dst), fr, rng, 5)                                    # restored event slot -> frame slot
    fr.finished()
    s = dst.restore([snaps[sl]])[0]                                          # -> restored event slot
    r = copy(rl)
    _serve(dst, s, r, rng, 5)
    r.finished()
    dst.free()


@gpu
@pytest.mark.parametrize("precision", [0, 1, 2])
def test_format(precision):
    """save(restore(b)) == b; SaveAny of frame-fed slots is Save's output byte for byte; SnapshotInfo and
    SnapshotEventInfo report counts and fg; blob == NULL sizing equals the written length."""
    g = _g()
    N = g._native
    ips = _voices(np.random.default_rng(150), 4)
    evs = [O.synthetic_event_list(151 + k, 0.3) for k in range(3)]
    fgs = [_fg("per-slot", k) for k in range(3)]
    fgs[1].reserved = 7                              # left non-zero by the caller: saved as 0, so it restores
    pushed = [0, 1, g.event_list_frame_count(evs[2])]
    a = g.TRMStreamPool(6, precision=precision, max_frames_per_push=80)
    ev_slots = [a.open_events(ips[k], evs[k], fgs[k])[0] for k in range(3)]
    fr_slots = [a.open(ips[3]), a.open(ips[0])]
    for s, k in zip(ev_slots, pushed):
        for at in range(0, k, 80):
            a.push({s: min(80, k - at)})
    a.push({fr_slots[0]: _walk(1, 17, seed=152)[0]})
    mixed = ev_slots + fr_slots
    snaps = a.save(mixed, event_slots=True)
    plain = a.save(fr_slots)
    for s in fr_slots:
        assert snaps[s] == plain[s] and g.snapshot_info(snaps[s])["events"] is None
    slot_a = np.array(mixed, np.int32)
    sized = np.zeros(len(mixed) + 1, np.int64)
    N.check(N.lib().TRMStreamPoolSaveAny(a._h, len(mixed), slot_a.ctypes.data_as(C.c_void_p), None, 0,
                                         sized.ctypes.data_as(C.c_void_p)), "size")
    blob = np.zeros(int(sized[-1]), np.uint8)
    written = np.zeros_like(sized)
    N.check(N.lib().TRMStreamPoolSaveAny(a._h, len(mixed), slot_a.ctypes.data_as(C.c_void_p), blob.ctypes.data_as(C.c_void_p),
                                         blob.size, written.ctypes.data_as(C.c_void_p)), "save")
    assert np.array_equal(sized, written)
    assert blob.tobytes() == b"".join(snaps[s] for s in mixed)
    b = g.TRMStreamPool(9, precision=precision, max_frames_per_push=3)
    b.open(ips[0])
    new = b.restore([snaps[s] for s in mixed])
    again = b.save(new, event_slots=True)
    for s, n in zip(mixed, new):
        assert again[n] == snaps[s]
    for k, s in enumerate(ev_slots):
        info = g.snapshot_info(snaps[s])
        assert info["precision"] == precision and info["frames_pushed"] == pushed[k] and info["bytes"] == len(snaps[s])
        e = info["events"]
        assert (e["n_events"], e["list_frames"], e["frames_generated"]) == (len(evs[k]), g.event_list_frame_count(evs[k]),
                                                                             pushed[k])
        for f, _ in fgs[k]._fields_:
            assert getattr(e["fg"], f) == (0 if f == "reserved" else getattr(fgs[k], f)), f
        assert struct.unpack_from("<i", snaps[s], FIXED + 60)[0] == 0
    a.free()
    b.free()


@gpu
def test_isolation_among_busy_slots():
    """300 busy slots, half event-fed, and one watched event slot: forks and migrations of busy event slots (their
    remaining frames read with snapshot_info) leave the watched slot and every busy request bit-identical to a run
    without them."""
    g = _g()
    ip = g.TRMInputParameters(44100.0, channels=2, balance=-0.4, volume=50.0)
    fg = g.TRMFrameGeneration()
    mine = O.synthetic_event_list(160, 0.2)
    nf = g.event_list_frame_count(mine)
    want = _events_one_shot(ip, mine, fg, 0)
    others = _voices(np.random.default_rng(161), 8)
    lists = [O.synthetic_event_list(1000 + i, 0.3) for i in range(150)]
    left0 = [g.event_list_frame_count(e) for e in lists]
    walks = _walk(150, 90, seed=162)

    def run(traffic):
        rng = np.random.default_rng(163)
        trng = np.random.default_rng(164)
        pool = g.TRMStreamPool(330, precision=0, max_frames_per_push=6)
        slot_of = {}
        for i in range(300):
            slot_of[i] = pool.open_events(others[i % 8], lists[i // 2], fg)[0] if i % 2 == 0 else pool.open(others[i % 8])
        s = pool.open_events(ip, mine, fg)[0]
        left = {i: left0[i // 2] for i in range(0, 300, 2)}
        wat = {i: 0 for i in range(1, 300, 2)}
        outs = {i: [] for i in range(300)}
        mine_out, at = [], 0
        forks = {}                                   # fork slot -> frames it has left
        while at < nf:
            m = min(4, nf - at)
            push = {s: m}
            for i in range(300):
                k = int(rng.integers(0, 7))
                if i % 2 == 0:
                    k = min(k, left[i])
                    left[i] -= k
                    push[slot_of[i]] = k
                else:
                    push[slot_of[i]] = walks[i // 2, wat[i]:wat[i] + k]
                    wat[i] += k
            for f in forks:
                k = min(int(trng.integers(0, 7)), forks[f])
                forks[f] -= k
                push[f] = k
            out = pool.push(push, flush={s} if at + m >= nf else ())
            mine_out.append(out[s])
            for i in range(300):
                outs[i].append(out[slot_of[i]])
            at += m
            if traffic:
                pick = [2 * int(x) for x in trng.choice(150, 6, replace=False)]
                snaps = pool.save([slot_of[i] for i in pick], event_slots=True)
                for n, i in zip(pool.restore([snaps[slot_of[i]] for i in pick[:3]]), pick[:3]):
                    e = g.snapshot_info(snaps[slot_of[i]])["events"]
                    forks[n] = e["list_frames"] - e["frames_generated"]
                for i in pick[3:]:
                    pool.close(slot_of[i])
                for i, n in zip(pick[3:], pool.restore([snaps[slot_of[i]] for i in pick[3:]])):
                    slot_of[i] = n
                while len(forks) > 12:
                    f = next(iter(forks))
                    pool.close(f)
                    del forks[f]
        pool.free()
        return np.concatenate(mine_out), {i: np.concatenate(outs[i]) for i in range(300)}

    quiet, noisy = run(False), run(True)
    _same(quiet[0], want[0], "watched slot, no snapshot traffic")
    _same(noisy[0], want[0], "watched slot among snapshot traffic")
    for i in range(300):
        _same(noisy[1][i], quiet[1][i], "busy request %d" % i)


def _set(b, at, fmt, value):
    b = bytearray(b)
    struct.pack_into(fmt, b, at, value)
    return _reseal(b)


def _add(b, at, fmt, delta):
    return _set(b, at, fmt, struct.unpack_from(fmt, b, at)[0] + delta)


@gpu
def test_refusals_leave_both_pools_unchanged():
    """Resealed changes to the generator's position, list_frames, n_events and the generator flag, a list with a track
    without later value, pending frames the destination's rows cannot take, another precision and too few free slots are
    refused; Save still refuses event slots.  After each refusal both pools' streams continue bit for bit."""
    g = _g()
    N = g._native
    rng = np.random.default_rng(170)
    ip = g.TRMInputParameters(44100.0)
    down = g.TRMInputParameters(22050.0, length=10.0, channels=2, balance=0.5)
    fg = g.TRMFrameGeneration()
    ev = O.synthetic_event_list(171, 0.5)
    a = g.TRMStreamPool(3, precision=0, max_frames_per_push=5)
    b = g.TRMStreamPool(3, precision=0, max_frames_per_push=4)
    ra, rb = EvRequest(0, ip, ev, fg, 0), EvRequest(1, down, O.synthetic_event_list(172, 0.5), fg, 0)
    walk = _walk(1, 60, seed=173)[0]
    rf = FrRequest(2, ip, walk, _frames_one_shot(ip, walk, 0))
    sa, sb, sf = ra.open(a), rb.open(b), rf.open(a)
    live = ((a, sa, ra), (b, sb, rb), (a, sf, rf))

    def step():
        for pool, s, r in live:
            r.got_samples(pool.push({s: r.take(max(0, min(3, r.nf - 6 - r.sent)))})[s])

    def refused(code, fn):
        with pytest.raises(g.TRMError) as e:
            fn()
        assert e.value.code == code, str(e.value)
        step()

    step()
    good = a.save([sa], event_slots=True)[sa]
    n_events, list_frames, generator = _ev_header(good)
    assert generator == 1
    at_gen = _at_gen(good)
    for off in (0, 8, 16):                                     # i, now, next
        refused(N.TRM_ERR_PARAM, lambda: b.restore([_add(good, at_gen + AT_GEN_I + off, "<q", 1)]))
    refused(N.TRM_ERR_PARAM, lambda: b.restore([_add(good, FIXED + 8, "<q", 1)]))          # list_frames
    refused(N.TRM_ERR_PARAM, lambda: b.restore([_add(good, FIXED + 8, "<q", -1)]))
    refused(N.TRM_ERR_PARAM, lambda: b.restore([_add(good, FIXED, "<q", -1)]))             # n_events vs the length
    refused(N.TRM_ERR_PARAM, lambda: b.restore([_add(good, FIXED, "<q", 1)]))
    refused(N.TRM_ERR_PARAM, lambda: b.restore([_set(good, FIXED + 64, "<I", 0)]))         # generator flag
    no_track = bytearray(good)                                 # track 4 has no value after the first event
    for k in range(1, n_events):
        struct.pack_into("<d", no_track, _at_list(good) + k * EVENT + 8 + 8 * 4, float("nan"))
    refused(N.TRM_ERR_PARAM, lambda: b.restore([_reseal(no_track)]))
    with pytest.raises(g.TRMError):
        g.snapshot_info(_reseal(no_track))

    # pending frames the rows cannot take: 18 generated frames all still pending (a consistent state Save never writes
    # at a control period of 8); pending rows hold max_frames_per_push + 16
    cp8 = _rate_voice(2500.0)
    p = g.TRMStreamPool(1, precision=0, max_frames_per_push=18)
    s = p.open_events(cp8, ev, fg)[0]
    p.push({s: 18})
    at18 = p.save([s], event_slots=True)[s]
    p.free()
    pend = _generated(ev, fg)[:18]
    big = (bytearray(at18[:AT_COUNTERS]) + struct.pack("<qqqqqii", 18, 0, 0, 0, 0, 18, 1) + at18[FIXED:FIXED + EVHEADER] +
           pend.tobytes() + at18[_at_gen(at18):])
    big = _reseal(big)
    assert g.snapshot_info(big)["events"]["frames_generated"] == 18
    refused(N.TRM_ERR_PARAM, lambda: b.restore([big]))

    # another precision, too few free slots, Save of an event slot
    p = g.TRMStreamPool(1, precision=2, max_frames_per_push=5)
    s = p.open_events(ip, ev, fg)[0]
    p.push({s: 5})
    other = p.save([s], event_slots=True)[s]
    p.free()
    refused(N.TRM_ERR_PARAM, lambda: b.restore([other]))
    refused(N.TRM_ERR_STATE, lambda: b.restore([good, good, good]))
    refused(N.TRM_ERR_STATE, lambda: a.save([sa]))
    refused(N.TRM_ERR_STATE, lambda: a.save([sf, sa]))
    two = b.restore([good, good])
    for s in two:
        b.close(s)
    for pool, s, r in live:
        _serve(pool, s, r, rng, pool.max_frames_per_push)
        r.finished()
    a.free()
    b.free()


# ---- no device needed ------------------------------------------------------------------------------------------------
def _position(ev, k):
    """framegen_step's (i, now, next) after k frames, stepped one frame at a time as the device does (the library computes
    it in O(events) instead): the clock advances 4 ms per frame; once it reaches the current event's time the next event
    becomes current, and `next` is left as it is when the last one is passed."""
    i, now, nxt = 1, 0, int(ev["time"][1]) & 0xFFFFFFFFFFFFFFFF
    for _ in range(k):
        now += 4
        if now >= nxt:
            i += 1
            if i == len(ev):
                break
            nxt = int(ev["time"][i]) & 0xFFFFFFFFFFFFFFFF
    return i, now, nxt


def _built_v2(ip, ev, fg, k=0, rng=None):
    """A version-2 snapshot written from the documented layout: the version-1 builder's header, voice and derived
    constants; counters of k generated frames that are all still pending (fresh); the event header; k pending frames,
    a generator state with the position k frames give (other fields random) and the list."""
    g = _g()
    v1 = _built_snapshot(ip)
    head = bytearray(v1[:AT_COUNTERS])
    struct.pack_into("<I", head, 8, 2)
    counters = struct.pack("<qqqqqii", k, 0, 0, 0, 0, k, 1)
    evh = struct.pack("<qq4idddfiII", len(ev), g.event_list_frame_count(ev), fg.useMacroIntonation, fg.useMicroIntonation,
                      fg.useSmoothIntonation, fg.useDrift, fg.driftDeviation, fg.driftCutoff, fg.pitch, fg.driftSeed, 0,
                      1 if k else 0, 0)
    assert len(evh) == EVHEADER
    data = b""
    if k:
        rng = rng or np.random.default_rng(k)
        data += rng.random((k, 16)).tobytes()
        data += rng.random(69).tobytes() + struct.pack("<qQQ", *_position(ev, k)) + rng.random(6).astype(np.float32).tobytes()
    assert len(data) == k * 128 + (GEN if k else 0)
    return _reseal(bytes(head) + counters + evh + data + ev.tobytes())


def test_version_2_layout_without_a_device():
    """SnapshotInfo and SnapshotEventInfo read version-2 snapshots written from the documented layout (never pushed, and
    with generated frames at event starts and in between); resealed changes to the event header or the generator's
    position, a version-2 body labelled version 1 and the reverse, and NULL arguments are refused."""
    g = _g()
    N = g._native
    L = N.lib()
    ip = g.TRMInputParameters(22050.0, length=10.0, channels=2, balance=0.25)
    fg = _fg("per-slot", 2)
    ev = O.synthetic_event_list(180, 0.8)
    nf = g.event_list_frame_count(ev)
    snap = _built_v2(ip, ev, fg)
    info = g.snapshot_info(snap)
    assert info["frames_pushed"] == 0 and info["bytes"] == FIXED + EVHEADER + len(ev) * EVENT
    e = info["events"]
    assert (e["n_events"], e["list_frames"], e["frames_generated"]) == (len(ev), nf, 0)
    for f, _ in fg._fields_:
        assert getattr(e["fg"], f) == getattr(fg, f), f
    st = _event_starts(ev)
    for k in (1, 2, st[0], st[0] + 1, st[3], (st[3] + st[4]) // 2, nf - 1, nf):
        b = _built_v2(ip, ev, fg, k)
        assert g.snapshot_info(b)["events"]["frames_generated"] == k
        at = _at_gen(b) + AT_GEN_I
        for off in (0, 8, 16):
            with pytest.raises(g.TRMError) as x:
                g.snapshot_info(_add(b, at + off, "<q", 1))
            assert x.value.code == N.TRM_ERR_PARAM, (k, off)
    with pytest.raises(g.TRMError):
        g.snapshot_info(_built_v2(ip, ev, fg, nf + 1))        # more frames than the list has
    for at, fmt, delta in ((FIXED, "<q", 1), (FIXED, "<q", -1), (FIXED + 8, "<q", 1), (FIXED + 8, "<q", -1),
                           (FIXED + 60, "<i", 1), (FIXED + 64, "<I", 1), (FIXED + 68, "<I", 1)):
        with pytest.raises(g.TRMError) as x:
            g.snapshot_info(_add(snap, at, fmt, delta))
        assert x.value.code == N.TRM_ERR_PARAM, (at, delta)
    with pytest.raises(g.TRMError):
        g.snapshot_info(_set(snap, 8, "<I", 1))                 # a version-2 body labelled version 1
    with pytest.raises(g.TRMError):
        g.snapshot_info(_set(_built_snapshot(ip), 8, "<I", 2))  # a version-1 body labelled version 2
    v1 = g.snapshot_info(_built_snapshot(ip))
    assert v1["events"] is None
    raw = N.TRMStreamSnapshotEventInfoStruct()
    raw.n_events = 5
    buf = C.create_string_buffer(_built_snapshot(ip), FIXED)
    assert L.TRMStreamPoolSnapshotEventInfo(buf, FIXED, C.byref(raw)) == 0 and raw.from_events == 0 and raw.n_events == 0
    assert L.TRMStreamPoolSnapshotEventInfo(None, 100, C.byref(raw)) == N.TRM_ERR_PARAM
    assert L.TRMStreamPoolSnapshotEventInfo(buf, FIXED, None) == N.TRM_ERR_PARAM
    off = np.zeros(2, np.int64)
    assert L.TRMStreamPoolSaveAny(None, 0, None, None, 0, off.ctypes.data_as(C.c_void_p)) == N.TRM_ERR_PARAM
