"""PCM16 pushes of the stream pool (TRMStreamPoolPushPCM16): a slot's new output scaled against a peak the caller gives
per push, in the slot's own channel layout, saturated to the int16 range.  With the utterance's maximumSampleValue as
the peak, a slot's PCM pushes, concatenated, equal the one-shot TRMBatch pcm_out bit for bit, and the maxima they
return reach that maximumSampleValue."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))

gpu = pytest.mark.gpu


def _g():
    import gnuspeech_b200 as g
    return g


def _one_shot(ips, frames, prec):
    """Whole utterances through TRMBatch: ips[u] with frames[u] ((nf, 16)) -> per utterance (samples, interleaved
    PCM16, maximumSampleValue)."""
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
    """The peak to scale against: the utterance's maximum (an all-zero utterance scales to zeros with any peak)."""
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
    """Stereo at balance +1, -1 and 0.3, mono and stereo at 60 dB (amplitude 1.0) and 42 dB, a 10 cm tract at 22.05 kHz
    (down-sampling), the female voice, then random voices."""
    g = _g()
    import fuzz_parity
    female = g.MMSynthesisParameters("Female").inputParameters()
    female.channels = 1
    vs = [g.TRMInputParameters(44100.0, channels=2, balance=1.0, volume=60.0),
          g.TRMInputParameters(44100.0, channels=2, balance=-1.0, volume=42.0),
          g.TRMInputParameters(44100.0, channels=2, balance=0.3, volume=60.0),
          g.TRMInputParameters(44100.0, channels=1, volume=42.0),
          g.TRMInputParameters(44100.0, channels=1, volume=60.0),
          g.TRMInputParameters(22050.0, length=10.0, channels=2, balance=0.3, volume=42.0),
          female]
    while len(vs) < n:
        vs.append(fuzz_parity.voice(rng))
    return vs[:n]


@gpu
@pytest.mark.parametrize("precision", [0, 1, 2])
def test_staggered_traffic_float_and_pcm_pushes(precision):
    """40 requests with different voices arrive at different pushes into a pool of 24 slots, advance by random frame
    counts and flush at different times; each push is randomly a float push or a PCM push.  A third of the requests
    are only ever advanced by PCM pushes."""
    g = _g()
    rng = np.random.default_rng(2000 + precision)
    n_req, cap, mmax = 40, 24, 12
    ips = _voices(rng, n_req)
    nfs = [int(x) for x in rng.integers(1, 70, n_req)]
    nfs[5] = 1                                       # a one-frame utterance: converter tail of silence only
    frames = [_walk(1, nf, seed=1300 + k)[0] for k, nf in enumerate(nfs)]
    want = _one_shot(ips, frames, precision)
    pcm_only = set(range(0, n_req, 3))
    start = sorted(int(x) for x in rng.integers(0, 25, n_req))
    pool = g.TRMStreamPool(cap, precision=precision, max_frames_per_push=mmax)
    waiting = list(range(n_req))
    active = {}                                      # slot -> [request, frames sent]
    pos = [0] * n_req                                # output samples returned so far
    mx = [0.0] * n_req                               # max over the request's PCM pushes
    kinds = set()
    t = 0
    while waiting or active:
        while waiting and start[waiting[0]] <= t and len(active) < cap:
            k = waiting.pop(0)
            active[pool.open(ips[k])] = [k, 0]
        as_pcm = bool(rng.random() < 0.5)
        kinds.add(as_pcm)
        push, flush = {}, set()
        for s, (k, at) in active.items():
            if rng.random() < 0.2 or (k in pcm_only and not as_pcm):
                continue                             # not named in this push
            m = min(int(rng.integers(0, mmax + 1)), nfs[k] - at)
            push[s] = frames[k][at:at + m]
            active[s][1] = at + m
            if at + m == nfs[k] and rng.random() < 0.7:
                flush.add(s)
        if as_pcm:
            out = pool.push_pcm16(push, {s: _peak(want[active[s][0]][2]) for s in set(push) | flush}, flush=flush)
            for s, (pcm, m) in out.items():
                k = active[s][0]
                ch = _channels(ips[k])
                assert pcm.dtype == np.int16 and pcm.shape[0] % ch == 0
                _same(pcm, want[k][1][pos[k] * ch:pos[k] * ch + pcm.shape[0]], "request %d, PCM push at %d" % (k, pos[k]))
                pos[k] += pcm.shape[0] // ch
                mx[k] = max(mx[k], m)
        else:
            out = pool.push(push, flush=flush)
            for s, y in out.items():
                k = active[s][0]
                _same(y, want[k][0][pos[k]:pos[k] + y.shape[0]], "request %d, float push at %d" % (k, pos[k]))
                pos[k] += y.shape[0]
        for s in flush:
            del active[s]
        t += 1
    pool.free()
    assert kinds == {False, True}
    for k in range(n_req):
        assert pos[k] == want[k][0].shape[0], ("request %d is incomplete" % k, pos[k], want[k][0].shape[0])
        assert mx[k] <= want[k][2], k
        if k in pcm_only:
            assert mx[k] == want[k][2], ("PCM-only request %d: max %r, maximumSampleValue %r" % (k, mx[k], want[k][2]))


@gpu
@pytest.mark.parametrize("precision", [0, 1, 2])
def test_saturation(precision):
    """At a peak of maximumSampleValue / 8 the PCM saturates at both bounds and never wraps: it equals
    clip(rint(y * scale)) of the one-shot samples, computed in float64 in the kernel's operation order."""
    g = _g()
    ips = [g.TRMInputParameters(44100.0, channels=1, volume=60.0),
           g.TRMInputParameters(44100.0, channels=2, balance=0.3, volume=60.0)]
    nf = 60
    frames = list(_walk(2, nf, seed=71))
    want = _one_shot(ips, frames, precision)
    pool = g.TRMStreamPool(2, precision=precision, max_frames_per_push=7)
    slots = [pool.open(ip) for ip in ips]
    peaks = {s: want[i][2] / 8 for i, s in enumerate(slots)}
    got, mx, at = [[], []], [0.0, 0.0], 0
    while at < nf:
        out = pool.push_pcm16({s: frames[i][at:at + 7] for i, s in enumerate(slots)}, peaks,
                              flush=set(slots) if at + 7 >= nf else ())
        for i, s in enumerate(slots):
            got[i].append(out[s][0])
            mx[i] = max(mx[i], out[s][1])
        at += 7
    pool.free()
    for i, ip in enumerate(ips):
        y = want[i][0].astype(np.float64)
        scale = (32767.0 / peaks[slots[i]]) * 1.0                # amplitude(60 dB) == 1.0
        if ip.channels == 2:
            b = ip.balance
            ls, rs = -((b / 2.0) - 0.5) * scale, ((b / 2.0) + 0.5) * scale
            raw = np.stack([np.rint(y * ls), np.rint(y * rs)], axis=1).reshape(-1)
        else:
            raw = np.rint(y * scale)
        ref = np.clip(raw, -32768, 32767).astype(np.int16)
        pcm = np.concatenate(got[i])
        _same(pcm, ref, "voice %d" % i)
        assert (raw > 32767).any() and (raw < -32768).any()
        assert (pcm == 32767).any() and (pcm == -32768).any()
        assert np.array_equal(pcm[raw > 32767], np.full(int((raw > 32767).sum()), 32767, np.int16))
        assert np.array_equal(pcm[raw < -32768], np.full(int((raw < -32768).sum()), -32768, np.int16))
        assert mx[i] == want[i][2]


@gpu
def test_isolation_among_busy_slots():
    """One stereo slot's PCM is the same alone and among 300 busy slots with other voices and peaks."""
    g = _g()
    rng = np.random.default_rng(13)
    ip = g.TRMInputParameters(44100.0, channels=2, balance=-0.4, volume=50.0)
    nf = 24
    mine = _walk(1, nf, seed=910)[0]
    want = _one_shot([ip], [mine], 0)[0]
    others = _voices(rng, 8)
    busy = _walk(300, nf, seed=911)

    def run(with_others):
        pool = g.TRMStreamPool(301, precision=0, max_frames_per_push=6)
        o = [pool.open(others[i % 8]) for i in range(300)] if with_others else []
        s = pool.open(ip)
        peaks = {so: float(rng.uniform(0.05, 2.0)) for so in o}
        peaks[s] = want[2]
        parts, at = [], 0
        oat = [0] * len(o)
        while at < nf:
            push = {s: mine[at:at + 4]}
            for i, so in enumerate(o):
                m = int(rng.integers(0, 7))
                push[so] = busy[i, oat[i]:oat[i] + m]
                oat[i] += m
            parts.append(pool.push_pcm16(push, peaks, flush={s} if at + 4 >= nf else ())[s][0])
            at += 4
        pool.free()
        return np.concatenate(parts)

    alone, among = run(False), run(True)
    _same(alone, want[1], "alone")
    _same(among, want[1], "among 300 busy slots")


@gpu
def test_refusals_leave_the_pool_unchanged():
    """Bad peaks and the float push's refusals, through the PCM call, change nothing: after each one a valid push
    continues, and the slots' PCM still equals the one-shot results."""
    g = _g()
    N = g._native
    ip = g.TRMInputParameters(44100.0)
    down = g.TRMInputParameters(22050.0, length=10.0, channels=2, balance=0.5)
    nf = 30
    frames = _walk(2, nf, seed=63)
    want = _one_shot([ip, down], list(frames), 0)
    pool = g.TRMStreamPool(3, precision=0, max_frames_per_push=5)
    a, b = pool.open(ip), pool.open(down)
    peaks = {a: want[0][2], b: want[1][2]}
    got = {0: [], 1: []}
    at = [0, 0]

    def step(flush=()):
        out = pool.push_pcm16({a: frames[0][at[0]:at[0] + 5], b: frames[1][at[1]:at[1] + 5]}, peaks, flush=flush)
        for s, i in ((a, 0), (b, 1)):
            got[i].append(out[s][0])
            at[i] += 5

    def refused(code, fn):
        with pytest.raises(g.TRMError) as e:
            fn()
        assert e.value.code == code

    def raw(slots, nfr, peak):
        """The C call with arguments the wrapper would not build (peak may be None: a NULL pointer)."""
        slot = np.array(slots, np.int32)
        nfr = np.array(nfr, np.int32)
        fr = np.ascontiguousarray(np.concatenate([frames[0][at[0]:at[0] + k] for k in nfr]))
        pk = None if peak is None else np.array(peak, np.float64)
        pcm = np.zeros(2 * len(slots) * pool.slot_capacity() + 1, np.int16)
        off = np.zeros(len(slots) + 1, np.int64)
        mx = np.zeros(len(slots), np.float64)
        vp = lambda x: None if x is None else x.ctypes.data_as(C.c_void_p)   # noqa: E731
        N.check(N.lib().TRMStreamPoolPushPCM16(pool._h, len(slots), vp(slot), vp(nfr), vp(fr), None, vp(pk), vp(pcm),
                                               vp(off), vp(mx)), "TRMStreamPoolPushPCM16")

    step()
    for bad in (0.0, -1.0, float("nan"), float("inf")):
        refused(N.TRM_ERR_PARAM, lambda: pool.push_pcm16({a: frames[0][at[0]:at[0] + 5], b: frames[1][at[1]:at[1] + 5]},
                                                         {a: peaks[a], b: bad}))
        step()
    refused(N.TRM_ERR_PARAM, lambda: raw([a], [5], None))                          # NULL peak
    refused(N.TRM_ERR_STATE, lambda: pool.push_pcm16({a: frames[0][at[0]:at[0] + 5], 2: frames[0][:5]}, 1.0))   # not open
    refused(N.TRM_ERR_PARAM, lambda: raw([a, a], [5, 5], [1.0, 1.0]))              # a slot named twice
    refused(N.TRM_ERR_PARAM, lambda: pool.push_pcm16({a: frames[0][:6]}, 1.0))                                    # 6 > max
    while at[0] < nf:
        step(flush={a, b} if at[0] + 5 >= nf else ())
    pool.free()
    for i in range(2):
        _same(np.concatenate(got[i]), want[i][1], "slot of utterance %d" % i)


def test_pcm_push_needs_a_pool():
    """A PCM push without a pool is refused (TRM_ERR_PARAM); this needs no device."""
    g = _g()
    N = g._native
    off = np.zeros(2, np.int64)
    assert N.lib().TRMStreamPoolPushPCM16(None, 0, None, None, None, None, None, None, off.ctypes.data_as(C.c_void_p),
                                          None) == N.TRM_ERR_PARAM
