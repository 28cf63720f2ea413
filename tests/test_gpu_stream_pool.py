"""Stream pool (TRMStreamPool): streaming slots that open, advance and end independently, each with its own voice.  The
contract is TRMStream's, per slot: a slot's concatenated output equals the one-shot TRMBatch synthesis of its utterance
with its voice, bit for bit, whatever the other slots do."""
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
    """Whole utterances through TRMBatch: ips[u] with frames[u] ((nf, 16)) -> list of sample arrays."""
    g = _g()
    b = g.TRMBatch(list(ips), [f.shape[0] for f in frames], precision=prec)
    smp = np.zeros(max(1, b.layout.total_out_samples), b.sample_dtype)
    b.synthesize(np.ascontiguousarray(np.concatenate(frames)), samples_out=smp, devices=[0])
    ns, oo = b.numberSamples, b.outOffsets
    return [smp[oo[u]:oo[u] + ns[u]].copy() for u in range(len(frames))]


def _same(got, want, what):
    assert got.shape == want.shape, (what, got.shape, want.shape)
    bad = ~((got == want) | (np.isnan(got) & np.isnan(want)))
    assert np.array_equal(got, want, equal_nan=True), "%s: %d samples differ, first at %d" % (
        what, int(bad.sum()), int(np.nonzero(bad)[0][0]))


def _walk(n, nf, seed):
    from gnuspeech_b200 import workloads as W
    return W.random_walk(n, nf, seed=seed).reshape(n, nf, 16)


def _voices(rng, n):
    """male 44.1 kHz, female, a 10 cm tract at 22.05 kHz (down-sampling), then random voices."""
    g = _g()
    import fuzz_parity
    female = g.MMSynthesisParameters("Female").inputParameters()
    female.channels = 1
    vs = [g.TRMInputParameters(44100.0), female, g.TRMInputParameters(22050.0, length=10.0)]
    while len(vs) < n:
        vs.append(fuzz_parity.voice(rng))
    return vs[:n]


@gpu
@pytest.mark.parametrize("precision", [0, 1, 2])
def test_staggered_traffic_with_mixed_voices(precision):
    """40 requests with different voices arrive at different pushes into a pool of 24 slots (so slots are reused), advance
    by random frame counts (0 .. max) and flush at different times."""
    g = _g()
    rng = np.random.default_rng(1000 + precision)
    n_req, cap, mmax = 40, 24, 12
    ips = _voices(rng, n_req)
    nfs = [int(x) for x in rng.integers(1, 70, n_req)]
    nfs[5] = 1                                       # a one-frame utterance: converter tail of silence only
    frames = [_walk(1, nf, seed=300 + k)[0] for k, nf in enumerate(nfs)]
    want = _one_shot(ips, frames, precision)
    start = sorted(int(x) for x in rng.integers(0, 25, n_req))
    pool = g.TRMStreamPool(cap, precision=precision, max_frames_per_push=mmax)
    waiting = list(range(n_req))
    active = {}                                      # slot -> [request, frames sent]
    got = [[] for _ in range(n_req)]
    t = 0
    while waiting or active:
        while waiting and start[waiting[0]] <= t and len(active) < cap:
            k = waiting.pop(0)
            active[pool.open(ips[k])] = [k, 0]
        push, flush = {}, set()
        for s, (k, at) in active.items():
            if rng.random() < 0.2:
                continue                             # not named in this push
            m = min(int(rng.integers(0, mmax + 1)), nfs[k] - at)
            push[s] = frames[k][at:at + m]
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
        _same(np.concatenate(got[k]) if got[k] else np.zeros(0, want[k].dtype), want[k], "request %d" % k)


@gpu
def test_different_sample_counts_in_one_cta():
    """Slots of one voice pushed together with a different frame count each: the pool sorts the slots by new samples and
    gives every CTA at least two of them, so each CTA holds utterances that end after different numbers of blocks -- the
    case in which a state saved when the CTA's loop ends would be wrong."""
    g = _g()
    n, pushes = 20, 6
    ip = g.TRMInputParameters(44100.0)
    counts = [[1 + (i * 7 + 3 * k) % n for i in range(n)] for k in range(pushes)]
    tot = [sum(counts[k][i] for k in range(pushes)) for i in range(n)]
    frames = [_walk(1, tot[i], seed=500 + i)[0] for i in range(n)]
    want = _one_shot([ip] * n, frames, 0)
    pool = g.TRMStreamPool(n, precision=0, max_frames_per_push=n)
    slots = [pool.open(ip) for _ in range(n)]
    got, at = [[] for _ in range(n)], [0] * n
    for k in range(pushes):
        push = {}
        for i, s in enumerate(slots):
            push[s] = frames[i][at[i]:at[i] + counts[k][i]]
            at[i] += counts[k][i]
        out = pool.push(push, flush=set(slots) if k == pushes - 1 else ())
        for i, s in enumerate(slots):
            got[i].append(out[s])
    pool.free()
    for i in range(n):
        _same(np.concatenate(got[i]), want[i], "slot %d" % i)


@gpu
@pytest.mark.parametrize("precision", [0, 1, 2])
def test_slot_reuse(precision):
    """A flushed slot reopened with another voice, and a slot closed in the middle of an utterance and reopened: the new
    utterance equals a fresh one-shot synthesis."""
    g = _g()
    rng = np.random.default_rng(7 + precision)
    ips = _voices(rng, 4)
    nf = [23, 31, 19, 27]
    frames = [_walk(1, nf[k], seed=700 + k)[0] for k in range(4)]
    want = _one_shot([ips[1], ips[2], ips[3]], frames[1:], precision)
    pool = g.TRMStreamPool(2, precision=precision, max_frames_per_push=8)
    a = pool.open(ips[0])
    b = pool.open(ips[1])
    got_b = [pool.push({a: frames[0][:8], b: frames[1][:8]})[b]]
    pool.close(a)                                    # client went away mid-utterance
    a2 = pool.open(ips[2])
    assert a2 == a
    got_a, at_a, at_b = [], 0, 8
    while at_b < nf[1]:
        out = pool.push({a2: frames[2][at_a:at_a + 5], b: frames[1][at_b:at_b + 8]}, flush={b} if at_b + 8 >= nf[1] else ())
        got_a.append(out[a2]); got_b.append(out[b])
        at_a += 5; at_b += 8
    b2 = pool.open(ips[3])                           # the flushed slot, another voice
    assert b2 == b
    got_c = []
    live = {a2: [2, at_a, 6, got_a], b2: [3, 0, 7, got_c]}      # slot -> [utterance, frames sent, per push, output]
    while live:
        push, fl = {}, set()
        for s, (k, at, m, _) in live.items():
            push[s] = frames[k][at:at + m]
            live[s][1] = at + m
            if at + m >= nf[k]:
                fl.add(s)
        out = pool.push(push, flush=fl)
        for s in push:
            live[s][3].append(out[s])
        for s in fl:
            del live[s]
    pool.free()
    _same(np.concatenate(got_b), want[0], "flushed slot")
    _same(np.concatenate(got_a), want[1], "reopened after close")
    _same(np.concatenate(got_c), want[2], "reopened after flush")


@gpu
def test_isolation_among_busy_slots():
    """One slot's output is the same alone and among 300 busy slots with other voices and push sizes."""
    g = _g()
    rng = np.random.default_rng(11)
    ip = g.MMSynthesisParameters("Female").inputParameters()
    ip.channels = 1
    nf = 24
    mine = _walk(1, nf, seed=900)[0]
    want = _one_shot([ip], [mine], 0)[0]
    others = _voices(rng, 8)
    busy = _walk(300, nf, seed=901)

    def run(with_others):
        pool = g.TRMStreamPool(301, precision=0, max_frames_per_push=6)
        o = [pool.open(others[i % 8]) for i in range(300)] if with_others else []
        s = pool.open(ip)
        parts, at = [], 0
        oat = [0] * len(o)
        while at < nf:
            push = {s: mine[at:at + 4]}
            for i, so in enumerate(o):
                m = int(rng.integers(0, 7))
                push[so] = busy[i, oat[i]:oat[i] + m]
                oat[i] += m
            parts.append(pool.push(push, flush={s} if at + 4 >= nf else ())[s])
            at += 4
        pool.free()
        return np.concatenate(parts)

    alone, among = run(False), run(True)
    _same(alone, want, "alone")
    _same(among, want, "among 300 busy slots")


@gpu
@pytest.mark.parametrize("case", ["walk_44k", "walk_short_tube_down"])
def test_slot_against_the_reference_float_stream(case):
    """The golden vectors hold the float stream Applications/TRAcT/tube.c emits for these frames; a slot fed them in small
    pushes, next to other slots, returns that stream to the float precision tube.c emits (2e-7 of peak)."""
    import oracle_lib as O
    g = _g()
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "trm_golden.npz"))
    oip = O.OracleInputParameters.from_buffer_copy(bytes(z[case + "/ip"]))
    frames = z[case + "/frames"]
    assert z[case + "/ref_agreement"][1] == 0.0
    ref_out = z[case + "/samples"].astype(np.float32)
    ip = g.TRMInputParameters(float(oip.outputRate))
    for name, _ in oip._fields_:
        if hasattr(ip, name):
            setattr(ip, name, getattr(oip, name))
    nf = frames.shape[0]
    other = _walk(3, nf, seed=41)
    pool = g.TRMStreamPool(4, precision=g.TRM_PRECISION_FP64, max_frames_per_push=16)
    o = [pool.open(v) for v in _voices(np.random.default_rng(3), 3)]
    s = pool.open(ip)
    parts, at = [], 0
    for m in ([5, 1, 16, 3] * nf)[:nf]:
        m = min(m, nf - at)
        if m <= 0:
            break
        push = {s: frames[at:at + m]}
        for i, so in enumerate(o):
            push[so] = other[i, at:at + (16 - m)]
        parts.append(pool.push(push, flush={s} if at + m >= nf else ())[s])
        at += m
    pool.free()
    y = np.concatenate(parts)
    assert y.shape[0] == ref_out.shape[0]
    peak = float(np.abs(ref_out).max())
    assert np.abs(y.astype(np.float32) - ref_out).max() <= 2e-7 * peak


@gpu
def test_errors_leave_the_pool_unchanged():
    """Refused calls change nothing: after each one a valid push continues, and the slots still equal their one-shot
    results."""
    g = _g()
    N = g._native
    ip = g.TRMInputParameters(44100.0)
    down = g.TRMInputParameters(22050.0, length=10.0)
    nf = 30
    frames = _walk(3, nf, seed=61)
    want = _one_shot([ip, down, ip], list(frames), 0)
    pool = g.TRMStreamPool(3, precision=0, max_frames_per_push=5)
    a, b = pool.open(ip), pool.open(down)
    got = {0: [], 1: [], 2: []}
    at = [0, 0, 0]

    def step(slots, idx, flush=()):
        out = pool.push({s: frames[i][at[i]:at[i] + 5] for s, i in zip(slots, idx)}, flush=flush)
        for s, i in zip(slots, idx):
            got[i].append(out[s])
            at[i] += 5

    def refused(code, fn):
        with pytest.raises(g.TRMError) as e:
            fn()
        assert e.value.code == code

    step([a, b], [0, 1])
    refused(N.TRM_ERR_STATE, lambda: pool.push({a: frames[0][5:10], 2: frames[2][:5]}))     # slot 2 is not open
    step([a, b], [0, 1])

    def duplicate():
        slot = np.array([a, a], np.int32)
        nfr = np.array([5, 5], np.int32)
        fr = np.ascontiguousarray(np.concatenate([frames[0][10:15], frames[0][15:20]]))
        out = np.zeros(2 * pool.slot_capacity() + 1, np.float64)
        off = np.zeros(3, np.int64)
        N.check(N.lib().TRMStreamPoolPush(pool._h, 2, slot.ctypes.data_as(C.c_void_p), nfr.ctypes.data_as(C.c_void_p),
                                          fr.ctypes.data_as(C.c_void_p), None, out.ctypes.data_as(C.c_void_p),
                                          off.ctypes.data_as(C.c_void_p)), "TRMStreamPoolPush")
    refused(N.TRM_ERR_PARAM, duplicate)
    refused(N.TRM_ERR_PARAM, lambda: pool.push({a: frames[0][10:16], b: frames[1][10:15]}))  # 6 > max_frames_per_push
    step([a, b], [0, 1])
    c = pool.open(ip)
    refused(N.TRM_ERR_STATE, lambda: pool.open(down))                                          # full
    small_cp = g.TRMInputParameters(44100.0)
    small_cp.controlRate = 5000.0                                                              # control period < 8
    low_ratio = g.TRMInputParameters(4000.0)                                                   # rate ratio below the staged rows
    for bad in (small_cp, low_ratio):
        with pytest.raises(g.TRMError):
            g.TRMBatch(bad, [10])
    pool.close(c)
    refused(N.TRM_ERR_PARAM, lambda: pool.open(small_cp))
    refused(N.TRM_ERR_PARAM, lambda: pool.open(low_ratio))
    c = pool.open(ip)
    while at[0] < nf:
        last = at[0] + 5 >= nf
        step([a, b, c], [0, 1, 2], flush={a, b} if last else ())
    while at[2] < nf:
        step([c], [2], flush={c} if at[2] + 5 >= nf else ())
    pool.free()
    for i in range(3):
        _same(np.concatenate(got[i]), want[i], "slot of utterance %d" % i)


def test_pool_needs_a_device():
    """Without a CUDA device there is no pool (no CPU fallback); a zero capacity is refused before any device is used."""
    g = _g()
    N = g._native
    err = C.c_int(0)
    assert not N.lib().TRMStreamPoolCreate(0, 0, 8, 0, C.byref(err))
    assert err.value == N.TRM_ERR_PARAM
    h = N.lib().TRMStreamPoolCreate(1, 0, 8, 0, C.byref(err))
    if h:
        N.lib().TRMStreamPoolFree(h)
        pytest.skip("a CUDA device is visible")
    assert err.value == N.TRM_ERR_CUDA
