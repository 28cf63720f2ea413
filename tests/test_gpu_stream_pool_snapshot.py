"""Stream pool snapshots (TRMStreamPoolSave / Restore / SnapshotInfo): a live slot saved to bytes and restored into any
pool of the same precision continues bit for bit.  A slot's output before the save, followed by the restored slot's
output, equals the one-shot TRMBatch synthesis of the utterance (samples, PCM at the utterance's peak, per-push maxima),
whatever either pool does.  Refused calls leave both pools exactly as they were."""
import ctypes as C
import os
import struct
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))

gpu = pytest.mark.gpu

# the snapshot layout include/trm.h documents
HEADER, VOICE, DERIVED, COUNTERS = 32, 192, 24, 48
FIXED = HEADER + VOICE + DERIVED + COUNTERS
AT_DERIVED, AT_COUNTERS = HEADER + VOICE, HEADER + VOICE + DERIVED


def _g():
    import gnuspeech_b200 as g
    return g


def _fnv1a64(b):
    h = 0xcbf29ce484222325
    for x in b:
        h = ((h ^ x) * 0x100000001b3) & 0xFFFFFFFFFFFFFFFF
    return h


def _counters(b):
    """(frames_seen, s_done, out_done, in_start, pend_first, pend_frames, fresh)"""
    return struct.unpack_from("<qqqqqii", b, AT_COUNTERS)


def _reseal(b):
    """b with its length and checksum fields made to match its bytes (for snapshots edited on purpose)"""
    b = bytearray(b)
    struct.pack_into("<Q", b, 16, len(b))
    struct.pack_into("<Q", b, 24, _fnv1a64(bytes(b[HEADER:])))
    return bytes(b)


def _one_shot(ips, frames, prec):
    """Whole utterances through TRMBatch -> per utterance (samples, interleaved PCM16, maximumSampleValue)."""
    g = _g()
    b = g.TRMBatch(list(ips), [f.shape[0] for f in frames], precision=prec)
    smp = np.zeros(max(1, b.layout.total_out_samples), b.sample_dtype)
    pcm = np.zeros(max(1, b.layout.total_pcm_samples), np.int16)
    b.synthesize(np.ascontiguousarray(np.concatenate(frames)), pcm_out=pcm, samples_out=smp, devices=[0])
    ns, oo, po, mx = b.numberSamples, b.outOffsets, b.pcmOffsets, b.maximumSampleValues
    return [(smp[oo[u]:oo[u] + ns[u]].copy(), pcm[po[u]:po[u] + ns[u] * _channels(ips[u])].copy(), float(mx[u]))
            for u in range(len(frames))]


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
    """Mono and stereo voices, the female voice, a 10 cm tract at 22.05 kHz (down-sampling), then random voices."""
    g = _g()
    import fuzz_parity
    female = g.MMSynthesisParameters("Female").inputParameters()
    female.channels = 1
    vs = [g.TRMInputParameters(44100.0), female, g.TRMInputParameters(22050.0, length=10.0),
          g.TRMInputParameters(44100.0, channels=2, balance=0.3, volume=60.0),
          g.TRMInputParameters(22050.0, length=10.0, channels=2, balance=-1.0, volume=42.0)]
    while len(vs) < n:
        vs.append(fuzz_parity.voice(rng))
    return vs[:n]


def _rate_voice(control_rate):
    """17.5 cm at 44.1 kHz: control rate 2500 Hz is a control period of 8, 1 Hz one of 19,794 tube samples."""
    ip = _g().TRMInputParameters(44100.0, length=17.5)
    ip.controlRate = control_rate
    return ip


def _fields(ip):
    return tuple(tuple(getattr(ip, f)) if f == "noseRadius" else getattr(ip, f) for f, _ in ip._fields_)


def _device_count():
    from gnuspeech_b200 import _native as N
    N.lib()
    return int(C.CDLL(N.LIBTRM_CUDA_PATH).trm_cuda_device_count())


class Request(object):
    """One utterance served by push after push, possibly through several slots and pools; checks every output as it
    arrives against the one-shot result."""

    def __init__(self, k, ip, frames, want, pcm_only=False):
        self.k, self.ip, self.frames, self.want, self.pcm_only = k, ip, frames, want, pcm_only
        self.sent = 0            # frames pushed so far
        self.pos = 0             # output samples returned so far
        self.mx = 0.0            # max over the PCM pushes' maxima

    def got_samples(self, y):
        _same(y, self.want[0][self.pos:self.pos + y.shape[0]], "request %d, float push at %d" % (self.k, self.pos))
        self.pos += y.shape[0]

    def got_pcm(self, pcm, m):
        ch = _channels(self.ip)
        assert pcm.shape[0] % ch == 0
        _same(pcm, self.want[1][self.pos * ch:self.pos * ch + pcm.shape[0]], "request %d, PCM push at %d" % (self.k, self.pos))
        self.pos += pcm.shape[0] // ch
        self.mx = max(self.mx, m)

    def finished(self):
        assert self.pos == self.want[0].shape[0], ("request %d is incomplete" % self.k, self.pos, self.want[0].shape[0])
        assert self.mx <= self.want[2]
        if self.pcm_only:
            assert self.mx == self.want[2], (self.k, self.mx, self.want[2])


def _push(pool, active, rng, mmax, as_pcm, p_skip=0.2):
    """One push of pool: every active request (slot -> Request) is named with prob. 1 - p_skip and advanced by 0..mmax
    frames; a request whose frames are all sent flushes with prob. 0.7.  Checks the outputs."""
    push, flush = {}, set()
    for s, r in active.items():
        if rng.random() < p_skip or (r.pcm_only and not as_pcm):
            continue
        m = min(int(rng.integers(0, mmax + 1)), r.frames.shape[0] - r.sent)
        push[s] = r.frames[r.sent:r.sent + m]
        r.sent += m
        if r.sent == r.frames.shape[0] and rng.random() < 0.7:
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
    """Saves each slot of src with prob. p (one Save call), closes them and restores the snapshots into dst (one Restore
    call), as far as dst has free slots.  Returns the number moved."""
    free = dst.capacity - len(dst_active)
    pick = [s for s in src_active if rng.random() < p][:free]
    if not pick:
        return 0
    snaps = src.save(pick)
    for s in pick:
        src.close(s)
    new = dst.restore([snaps[s] for s in pick])
    assert len(set(new)) == len(new) and not set(new) & set(dst_active)
    for s, n in zip(pick, new):
        dst_active[n] = src_active.pop(s)
    return len(pick)


def _traffic(precision, dev_b, seed):
    """Staggered traffic over two pools of different capacity and max_frames_per_push (the second on device dev_b):
    requests open in the first, live slots migrate both ways at random push boundaries, float and PCM pushes mix."""
    g = _g()
    rng = np.random.default_rng(seed)
    n_req = 40
    ips = _voices(rng, n_req)
    nfs = [int(x) for x in rng.integers(1, 70, n_req)]
    nfs[5] = 1
    frames = [_walk(1, nf, seed=seed * 7 + k)[0] for k, nf in enumerate(nfs)]
    want = _one_shot(ips, frames, precision)
    reqs = [Request(k, ips[k], frames[k], want[k], pcm_only=(k % 3 == 0)) for k in range(n_req)]
    start = sorted(int(x) for x in rng.integers(0, 25, n_req))
    a = g.TRMStreamPool(24, precision=precision, max_frames_per_push=12)
    b = g.TRMStreamPool(17, precision=precision, max_frames_per_push=9, device=dev_b)
    a_act, b_act = {}, {}
    waiting = list(range(n_req))
    moved, t = 0, 0
    while waiting or a_act or b_act:
        while waiting and start[waiting[0]] <= t and len(a_act) < a.capacity:
            k = waiting.pop(0)
            a_act[a.open(ips[k])] = reqs[k]
        _push(a, a_act, rng, a.max_frames_per_push, bool(rng.random() < 0.5))
        _push(b, b_act, rng, b.max_frames_per_push, bool(rng.random() < 0.5))
        moved += _migrate(rng, a, a_act, b, b_act, 0.15)
        moved += _migrate(rng, b, b_act, a, a_act, 0.05)
        t += 1
    a.free()
    b.free()
    for r in reqs:
        r.finished()
    assert moved >= 20, moved
    return moved


@gpu
@pytest.mark.parametrize("precision", [0, 1, 2])
def test_migration_under_staggered_traffic(precision):
    _traffic(precision, 0, 4000 + precision)


@gpu
@pytest.mark.parametrize("precision", [0, 1, 2])
def test_migration_across_devices(precision):
    if _device_count() < 2:
        pytest.skip("one CUDA device: the second pool of the migration test would be on the same device")
    _traffic(precision, 1, 4100 + precision)


@gpu
@pytest.mark.parametrize("precision", [0, 1, 2])
def test_fork(precision):
    """A slot saved after a prefix and restored three times into the same pool: the source and the copies continue with
    different frames (two copies from the same snapshot with the same frames), and one copy is forked again.  Every
    branch equals the one-shot synthesis of its own frames."""
    g = _g()
    rng = np.random.default_rng(50 + precision)
    ip = g.TRMInputParameters(22050.0, length=10.0, channels=2, balance=0.3)
    pre, n_cont = 23, 31
    prefix = _walk(1, pre, seed=60)[0]
    conts = list(_walk(5, n_cont, seed=61))
    pool = g.TRMStreamPool(8, precision=precision, max_frames_per_push=7)
    s0 = pool.open(ip)
    head, at = [], 0
    while at < pre:
        m = int(rng.integers(1, 8))
        head.append(pool.push({s0: prefix[at:at + m]})[s0])
        at += m
    head = np.concatenate(head)
    snap = pool.save([s0])[s0]
    c1, c2, c3 = pool.restore([snap, snap, snap])
    # branch: slot -> (frames after the prefix, outputs after the prefix)
    br = {s0: [conts[0], []], c1: [conts[1], []], c2: [conts[1], []], c3: [conts[2], []]}
    sent = {s: 0 for s in br}

    def step(slots, m):
        push = {s: br[s][0][sent[s]:min(sent[s] + m, n_cont)] for s in slots}
        flush = {s for s in slots if sent[s] + m >= n_cont}
        for s, y in pool.push(push, flush=flush).items():
            br[s][1].append(y)
        for s in slots:
            sent[s] += m

    step(list(br), 5)
    step(list(br), 6)
    # fork of the fork: c3 after 11 of its own frames continues as c4 with other frames
    c4 = pool.restore([pool.save([c3])[c3]])[0]
    br[c4] = [np.concatenate([conts[2][:11], conts[3]]), [np.zeros(0, pool.dtype)]]
    sent[c4] = 11
    c4_head = np.concatenate(br[c3][1])
    while any(sent[s] < n_cont for s in br):
        step([s for s in br if sent[s] < n_cont], 7)
    pool.free()
    wanted = [np.concatenate([prefix, br[s][0][:n_cont]]) for s in (s0, c1, c3)] + [np.concatenate([prefix, br[c4][0][:n_cont]])]
    want = _one_shot([ip] * 4, wanted, precision)
    got = {s: np.concatenate([head] + br[s][1]) for s in br}
    _same(got[s0], want[0][0], "source")
    _same(got[c1], want[1][0], "copy 1")
    _same(got[c2], got[c1], "copy 2 (same snapshot, same frames)")
    _same(got[c3], want[2][0], "copy 3")
    _same(np.concatenate([head, c4_head] + br[c4][1]), want[3][0], "fork of copy 3")


def _serve(pool, slot, r, rng, mmax, pcm_every=2):
    """Pushes r's remaining frames through slot and flushes; alternates float and PCM pushes."""
    k = 0
    while True:
        m = min(int(rng.integers(1, mmax + 1)), r.frames.shape[0] - r.sent)
        last = r.sent + m == r.frames.shape[0]
        fr = {slot: r.frames[r.sent:r.sent + m]}
        r.sent += m
        if k % pcm_every:
            pcm, mx = pool.push_pcm16(fr, _peak(r.want[2]), flush={slot} if last else ())[slot]
            r.got_pcm(pcm, mx)
        else:
            r.got_samples(pool.push(fr, flush={slot} if last else ())[slot])
        k += 1
        if last:
            return


@gpu
@pytest.mark.parametrize("precision", [0, 1, 2])
def test_edge_states(precision):
    """Snapshots of a slot opened and never pushed, of a slot with one frame (fresh, pending frames only), taken inside a
    control interval, at control periods 8 and 19,794; restored into a pool whose rows and SlotCapacity must grow."""
    g = _g()
    rng = np.random.default_rng(70 + precision)
    male = g.TRMInputParameters(44100.0)
    cp8, cp19794 = _rate_voice(2500.0), _rate_voice(1.0)
    assert g.derive(cp8, 2).controlPeriod == 8 and g.derive(cp19794, 2).controlPeriod == 19794
    cases = [("never pushed", male, 30, 0), ("one frame", male, 30, 1), ("mid interval", male, 40, 13),
             ("period 8", cp8, 300, 157), ("period 19794", cp19794, 7, 3)]
    frames = [_walk(1, nf, seed=80 + i)[0] for i, (_, _, nf, _) in enumerate(cases)]
    want = _one_shot([c[1] for c in cases], frames, precision)
    a = g.TRMStreamPool(len(cases), precision=precision, max_frames_per_push=5)
    reqs, slots = [], []
    for i, (name, ip, nf, before) in enumerate(cases):
        r = Request(i, ip, frames[i], want[i])
        s = a.open(ip)
        while r.sent < before:
            m = min(5, before - r.sent)
            r.got_samples(a.push({s: frames[i][r.sent:r.sent + m]})[s])
            r.sent += m
        reqs.append(r)
        slots.append(s)
    snaps = a.save(slots)
    c = {name: _counters(snaps[s]) for (name, _, _, _), s in zip(cases, slots)}
    assert c["never pushed"] == (0, 0, 0, 0, 0, 0, 1)
    assert c["one frame"] == (1, 0, 0, 0, 0, 1, 1)
    fs, s_done, out_done, in_start, pend_first, pend_frames, fresh = c["mid interval"]
    assert fresh == 0 and s_done % 79 != 0 and pend_frames >= 2 and out_done > 0
    assert c["period 8"][1] > 0 and c["period 19794"][1] % 19794 != 0
    for s in slots:
        a.close(s)
    # the destination was sized for the default voice and 2 frames per push: the 19,794-sample period widens it
    b = g.TRMStreamPool(len(cases) + 3, precision=precision, max_frames_per_push=2)
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
def test_format_round_trip_and_info(precision):
    """save(restore(b)) == b byte for byte, in another pool and at another slot; snapshot_info reports the voice, the
    precision and the counts of real snapshots."""
    g = _g()
    ips = _voices(np.random.default_rng(90), 6)
    frames = list(_walk(6, 40, seed=91))
    pushed = [0, 1, 5, 17, 29, 40]
    a = g.TRMStreamPool(6, precision=precision, max_frames_per_push=40)
    slots = [a.open(ip) for ip in ips]
    returned = {}
    for s, k, fr in zip(slots, pushed, frames):
        returned[s] = a.push({s: fr[:k]})[s].shape[0] if k else 0
    snaps = a.save(slots)
    b = g.TRMStreamPool(9, precision=precision, max_frames_per_push=3)
    b.open(ips[0])                                   # the copies land at other slot numbers
    new = b.restore([snaps[s] for s in slots])
    assert new != slots
    again = b.save(new)
    for s, n, ip, k in zip(slots, new, ips, pushed):
        assert again[n] == snaps[s]
        info = g.snapshot_info(snaps[s])
        assert info["precision"] == precision and info["bytes"] == len(snaps[s])
        assert info["channels"] == _channels(ip)
        assert info["frames_pushed"] == k and info["samples_returned"] == returned[s]
        assert _fields(info["voice"]) == _fields(ip)
    a.free()
    b.free()


@gpu
def test_isolation_among_busy_slots():
    """300 busy slots and one watched slot: saves, forks, migrations and closes of busy slots inside the pool leave the
    watched slot and every busy request bit-identical to a run without them."""
    g = _g()
    ip = g.TRMInputParameters(44100.0, channels=2, balance=-0.4, volume=50.0)
    nf = 24
    mine = _walk(1, nf, seed=910)[0]
    want = _one_shot([ip], [mine], 0)[0]
    others = _voices(np.random.default_rng(13), 8)
    busy = _walk(300, nf + 6 * 6, seed=911)

    def run(traffic):
        rng = np.random.default_rng(14)             # the same frame counts in both runs
        trng = np.random.default_rng(15)
        pool = g.TRMStreamPool(340, precision=0, max_frames_per_push=6)
        slot_of = {i: pool.open(others[i % 8]) for i in range(300)}
        s = pool.open(ip)
        outs = {i: [] for i in range(300)}
        mine_out, at = [], 0
        oat = [0] * 300
        forks = []
        while at < nf:
            push = {s: mine[at:at + 4]}
            for i in range(300):
                m = int(rng.integers(0, 7))
                push[slot_of[i]] = busy[i, oat[i]:oat[i] + m]
                oat[i] += m
            for f in forks:
                push[f] = busy[0, :int(trng.integers(0, 7))]
            out = pool.push(push, flush={s} if at + 4 >= nf else ())
            mine_out.append(out[s])
            for i in range(300):
                outs[i].append(out[slot_of[i]])
            at += 4
            if traffic:
                pick = [int(x) for x in trng.choice(300, 6, replace=False)]
                snaps = pool.save([slot_of[i] for i in pick])
                forks += pool.restore([snaps[slot_of[i]] for i in pick[:3]])          # forks, pushed with other frames
                for i in pick[3:]:                                                     # migrations inside the pool
                    pool.close(slot_of[i])
                for i, n in zip(pick[3:], pool.restore([snaps[slot_of[i]] for i in pick[3:]])):
                    slot_of[i] = n
                while len(forks) > 12:
                    pool.close(forks.pop(0))
        pool.free()
        return np.concatenate(mine_out), {i: np.concatenate(outs[i]) for i in range(300)}

    quiet, noisy = run(False), run(True)
    _same(quiet[0], want[0], "watched slot, no snapshot traffic")
    _same(noisy[0], want[0], "watched slot among snapshot traffic")
    for i in range(300):
        _same(noisy[1][i], quiet[1][i], "busy request %d" % i)


@gpu
def test_refusals_leave_both_pools_unchanged():
    """Corrupt snapshots, other precisions, too few free slots, a snapshot whose pending frames would not fit the next
    push, and bad Save arguments are refused; after each refusal both pools' streams continue bit for bit."""
    g = _g()
    N = g._native
    rng = np.random.default_rng(99)
    ips = [g.TRMInputParameters(44100.0), g.TRMInputParameters(22050.0, length=10.0, channels=2, balance=0.5)]
    nf = 60
    frames = list(_walk(2, nf, seed=98))
    want = _one_shot(ips, frames, 0)
    a = g.TRMStreamPool(3, precision=0, max_frames_per_push=5)
    b = g.TRMStreamPool(3, precision=0, max_frames_per_push=4)
    ra, rb = Request(0, ips[0], frames[0], want[0]), Request(1, ips[1], frames[1], want[1])
    sa, sb = a.open(ips[0]), b.open(ips[1])

    def step():
        for pool, s, r in ((a, sa, ra), (b, sb, rb)):
            m = min(3, nf - 3 - r.sent)                  # the last 3 frames are left for the end
            r.got_samples(pool.push({s: r.frames[r.sent:r.sent + m]})[s])
            r.sent += m

    def refused(code, fn):
        with pytest.raises(g.TRMError) as e:
            fn()
        assert e.value.code == code, str(e.value)
        step()

    step()
    good = a.save([sa])[sa]
    flipped = bytearray(good)
    flipped[FIXED + 40] ^= 0x10
    refused(N.TRM_ERR_PARAM, lambda: b.restore([bytes(flipped)]))
    refused(N.TRM_ERR_PARAM, lambda: b.restore([good[:-8]]))
    refused(N.TRM_ERR_PARAM, lambda: b.restore([good[:20]]))
    wrong_version = bytearray(good)
    struct.pack_into("<I", wrong_version, 8, 2)
    refused(N.TRM_ERR_PARAM, lambda: b.restore([bytes(wrong_version)]))
    derived = bytearray(good)                            # a control period another build might derive
    struct.pack_into("<I", derived, AT_DERIVED, struct.unpack_from("<I", derived, AT_DERIVED)[0] + 1)
    refused(N.TRM_ERR_PARAM, lambda: b.restore([_reseal(derived)]))
    counters = bytearray(good)                           # a kept history that starts after what the converter reads
    struct.pack_into("<q", counters, AT_COUNTERS + 24, _counters(good)[1])
    refused(N.TRM_ERR_PARAM, lambda: b.restore([_reseal(counters)]))
    with pytest.raises(g.TRMError):
        g.snapshot_info(bytes(flipped))

    # other precisions: strict -> conformance (same element size), FP32 -> FP64
    for prec in (2, 1):
        p = g.TRMStreamPool(1, precision=prec, max_frames_per_push=5)
        s = p.open(ips[0])
        p.push({s: frames[0][:5]})
        other = p.save([s])[s]
        p.free()
        assert g.snapshot_info(other)["precision"] == prec
        refused(N.TRM_ERR_PARAM, lambda: b.restore([other]))

    # too few free slots: b has 2 free, 3 snapshots restore nothing
    refused(N.TRM_ERR_STATE, lambda: b.restore([good, good, good]))
    two = b.restore([good, good])
    refused(N.TRM_ERR_STATE, lambda: b.restore([good]))
    for s in two:
        b.close(s)

    # a snapshot with 40 pending frames and no synthesized sample (a state Save never writes, but a consistent one):
    # the next push synthesizes all of them.  It fits a pool whose rows were widened for a 1 Hz voice, not b.
    p = g.TRMStreamPool(2, precision=0, max_frames_per_push=4)
    s = p.open(ips[0])
    p.push({s: frames[0][:1]})
    one = p.save([s])[s]
    p.free()
    fs, s_done, out_done, in_start, pend_first, pend_frames, fresh = _counters(one)
    assert (fs, s_done, pend_frames, fresh) == (1, 0, 1, 1)
    k = 40
    big = bytearray(one[:AT_COUNTERS]) + struct.pack("<qqqqqii", k, 0, 0, 0, 0, k, 1) + frames[0][:k].tobytes()
    big = _reseal(big)
    assert g.snapshot_info(big)["frames_pushed"] == k
    refused(N.TRM_ERR_PARAM, lambda: b.restore([big]))
    wide = g.TRMStreamPool(2, precision=0, max_frames_per_push=4)
    wide.close(wide.open(_rate_voice(1.0)))
    rw = Request(2, ips[0], frames[0], want[0])
    rw.sent = k
    _serve(wide, wide.restore([big])[0], rw, rng, 4)
    rw.finished()
    wide.free()

    # Save: an unopened slot, a slot named twice, a buffer too small
    refused(N.TRM_ERR_STATE, lambda: a.save([sa, 2]))
    slot2 = np.array([sa, sa], np.int32)
    off = np.zeros(3, np.int64)
    refused(N.TRM_ERR_PARAM, lambda: N.check(N.lib().TRMStreamPoolSave(a._h, 2, slot2.ctypes.data_as(C.c_void_p), None, 0,
                                                                        off.ctypes.data_as(C.c_void_p)), "save"))
    slot1 = np.array([sa], np.int32)
    N.check(N.lib().TRMStreamPoolSave(a._h, 1, slot1.ctypes.data_as(C.c_void_p), None, 0, off.ctypes.data_as(C.c_void_p)), "size")
    small = np.zeros(int(off[1]) - 1, np.uint8)
    refused(N.TRM_ERR_PARAM, lambda: N.check(N.lib().TRMStreamPoolSave(a._h, 1, slot1.ctypes.data_as(C.c_void_p),
                                                                        small.ctypes.data_as(C.c_void_p), small.size,
                                                                        off.ctypes.data_as(C.c_void_p)), "save"))
    for pool, s, r in ((a, sa, ra), (b, sb, rb)):
        _serve(pool, s, r, rng, pool.max_frames_per_push)
        r.finished()
    a.free()
    b.free()


# ---- no device needed ------------------------------------------------------------------------------------------------
def _built_snapshot(ip, precision=0):
    """The snapshot of a slot opened with `ip` and never pushed, written from the documented layout: header, voice field by
    field, derived constants, counters, no data."""
    g = _g()
    dv = g.derive(ip, 2)
    voice = struct.pack("<iffdidi" + "d" * 10 + "d" * 6 + "ddid", ip.outputFileFormat, ip.outputRate, ip.controlRate,
                        ip.volume, ip.channels, ip.balance, ip.waveform, ip.tp, ip.tnMin, ip.tnMax, ip.breathiness,
                        ip.length, ip.temperature, ip.lossFactor, ip.apScale, ip.mouthCoef, ip.noseCoef,
                        *list(ip.noseRadius), ip.throatCutoff, ip.throatVol, ip.usesModulation, ip.mixOffset)
    assert len(voice) == VOICE
    derived = struct.pack("<6I", dv.controlPeriod, dv.sampleRate, dv.timeRegisterIncrement, dv.padSize, ip.channels,
                          4 if precision == 1 else 8)
    counters = struct.pack("<qqqqqii", 0, 0, 0, 0, 0, 0, 1)
    head = b"TRMSNAP\0" + struct.pack("<IIQQ", 1, precision, 0, 0)
    return _reseal(head + voice + derived + counters)


def test_snapshot_info_refuses_bad_input():
    """SnapshotInfo refuses NULL, short and garbage input, a changed derived constant and counters that disagree, and
    reads a snapshot written from the documented layout; Save and Restore refuse a NULL pool.  No device is used."""
    g = _g()
    N = g._native
    L = N.lib()
    info = N.TRMStreamSnapshotInfoStruct()
    assert L.TRMStreamPoolSnapshotInfo(None, 100, C.byref(info)) == N.TRM_ERR_PARAM
    short = C.create_string_buffer(b"TRMSNAP\0\1\0\0\0", 12)
    assert L.TRMStreamPoolSnapshotInfo(short, 12, C.byref(info)) == N.TRM_ERR_PARAM
    garbage = np.random.default_rng(5).integers(0, 256, 400).astype(np.uint8).tobytes()
    assert L.TRMStreamPoolSnapshotInfo(C.create_string_buffer(garbage, 400), 400, C.byref(info)) == N.TRM_ERR_PARAM
    ip = g.TRMInputParameters(22050.0, length=10.0, channels=2, balance=0.25)
    snap = _built_snapshot(ip)
    got = g.snapshot_info(snap)
    assert got["precision"] == 0 and got["channels"] == 2 and got["frames_pushed"] == 0 and got["bytes"] == FIXED
    assert _fields(got["voice"]) == _fields(ip)
    assert g.snapshot_info(_built_snapshot(ip, 1))["precision"] == 1
    for at, fmt, delta in ((AT_DERIVED, "<I", 1), (AT_DERIVED + 8, "<I", 1), (AT_COUNTERS, "<q", 1), (AT_COUNTERS + 44, "<i", -1)):
        bad = bytearray(snap)
        struct.pack_into(fmt, bad, at, struct.unpack_from(fmt, bad, at)[0] + delta)
        with pytest.raises(g.TRMError) as e:
            g.snapshot_info(_reseal(bad))
        assert e.value.code == N.TRM_ERR_PARAM
    tampered = bytearray(snap)
    tampered[HEADER + 12] ^= 1                          # the voice's volume, checksum left as it was
    with pytest.raises(g.TRMError):
        g.snapshot_info(bytes(tampered))
    bad_voice = g.TRMInputParameters(44100.0, channels=3)
    with pytest.raises(g.TRMError):
        g.snapshot_info(_built_snapshot(bad_voice))
    off = np.zeros(2, np.int64)
    assert L.TRMStreamPoolSave(None, 0, None, None, 0, off.ctypes.data_as(C.c_void_p)) == N.TRM_ERR_PARAM
    assert L.TRMStreamPoolRestore(None, 0, None, off.ctypes.data_as(C.c_void_p), None) == N.TRM_ERR_PARAM
