"""The resampler at the output rates the API accepts: ratio 1, either side of it, the down-sampling bound and high
up-sampling, in the batch, stream and pool paths.

Almost all of the converter's geometry follows from the ratio outputRate / tube rate: the pad (13 when up-sampling,
floor(13 / (65536 / tri)) + 1 when down-sampling), the time-register increment tri, the phase increment, the outputs
per work item nt (trm_cuda.cu plan_chunk), the work item's window of staged rows, the taps per filter wing of the
down-sampling phase walk (ceil(13 * 65536 / phaseIncrement)), what a stream or pool slot may emit and keeps as history,
and a pool's row width.  RATES holds one voice per edge of those formulas, at tube rates 19,750, 17,500, 18,000 and
35,000 Hz; every test below uses it.  `geometry()` gives each entry's (tube rate, outputRate, tri, phaseIncrement,
pad, nt), and `test_rate_table_hits_its_cases` proves the table holds each case."""
import ctypes as C
import math
import time

import numpy as np
import pytest

import oracle_lib as O

gpu = pytest.mark.gpu

FP64_TOL = 1e-9
FP32_SNR_DB = 80.0
SRC_ROWS, NT_MAX, SRC_CHUNK, SRC_WARPS = 128, 192, 8, 8      # include/trm_cuda.h, src_kernel.cuh SrcCfg, kernel_args.h

# (case, tract length in cm, outputRate, other voice fields).  Tube rates: 17.5 cm -> 19,750 Hz, 19.8 cm -> 17,500 Hz,
# 19.24 cm -> 18,000 Hz, 9.9 cm -> 35,000 Hz (control rate 250 Hz, 25 C).
RATES = [
    ("ratio 1", 17.5, 19750.0, {}),
    ("tri 65536 from below", 17.5, 19749.9, {}),            # down-sampling, phase increment 65536, pad 14
    ("tri 65536 from above", 17.5, 19750.1, dict(channels=2, balance=0.3)),
    ("just below 1", 17.5, 19749.0, {}),                     # tri 65539, phase increment 65533, pad 14
    ("just above 1", 17.5, 19751.0, {}),
    ("just above 1", 17.5, 19769.0, {}),
    ("bound", 17.5, 5463.0, {}),                             # the lowest accepted rate: pad 47, nt 8
    ("pad + 1 taps", 17.5, 5971.0, dict(channels=2, balance=-0.5)),
    ("48 kHz", 17.5, 48000.0, {}),
    ("96 kHz", 17.5, 96000.0, {}),
    ("192 kHz", 17.5, 192000.0, dict(channels=2, balance=0.7)),
    ("bound", 19.8, 4841.0, {}),
    ("pad + 1 taps", 19.8, 8125.0, {}),
    ("pad + 1 taps", 19.8, 6894.0, {}),
    ("44.1 kHz", 19.8, 44100.0, {}),
    ("pad + 1 taps", 19.24, 10174.0, {}),
    ("bound", 19.24, 4979.0, dict(channels=2, balance=0.0)),
    ("ratio 1", 9.9, 35000.0, {}),
    ("bound", 9.9, 9681.0, {}),
    ("192 kHz", 9.9, 192000.0, {}),
]
TUBE_RATES = {17.5: 19750, 19.8: 17500, 19.24: 18000, 9.9: 35000}


def _g():
    import gnuspeech_b200 as g
    return g


def voice(k):
    """TRMInputParameters of RATES[k]: Monet's male voice at that tract length and output rate"""
    _, length, out_rate, kw = RATES[k]
    return _g().TRMInputParameters(out_rate, length=length, **kw)


def geometry(k):
    """the converter geometry of RATES[k], as libtrm derives it and plan_chunk sizes its work items"""
    ip = voice(k)
    d = _g().derive(ip, 2)
    tri, pad = d.timeRegisterIncrement, d.padSize
    ratio = float(ip.outputRate) / d.sampleRate
    up = ratio >= 1.0
    unit = SRC_CHUNK * SRC_WARPS if up else SRC_CHUNK
    nt = min(int((SRC_ROWS - 3 - 2 * (pad + 1)) * 65536.0 / tri), NT_MAX) // unit * unit
    return dict(case=RATES[k][0], tube_rate=d.sampleRate, outputRate=float(ip.outputRate), ratio=ratio, up=up, tri=tri,
                phaseIncrement=0 if up else int(round(ratio * 65536.0)), pad=pad, nt=nt)


def describe(k):
    s = geometry(k)
    return "%s (tube %d Hz, outputRate %g, tri %d, phaseIncrement %d, pad %d, nt %d)" % (
        s["case"], s["tube_rate"], s["outputRate"], s["tri"], s["phaseIncrement"], s["pad"], s["nt"])


def entries(case):
    return [k for k, r in enumerate(RATES) if r[0] == case]


def accepted(out_rate, length):
    """TRMBatchCreate's answer for a voice: True, or the error code it refused the voice with"""
    g = _g()
    try:
        g.TRMBatch(g.TRMInputParameters(float(out_rate), length=length), [3])
        return True
    except g.TRMError as e:
        return e.code


def lowest_accepted_rate(length):
    """bisection on integer output rates: the lowest one TRMBatchCreate accepts for this tract length"""
    lo, hi = 1000, TUBE_RATES[length]
    assert accepted(lo, length) is not True and accepted(hi, length) is True
    while hi - lo > 1:
        mid = (lo + hi) // 2
        if accepted(mid, length) is True:
            hi = mid
        else:
            lo = mid
    return hi


def _walk(nf, seed):
    from gnuspeech_b200 import workloads as W
    return np.ascontiguousarray(W.random_walk(1, nf, seed=seed))


def _frames_off_nt(nf, k):
    """the smallest frame count >= nf whose output count is not a multiple of the entry's nt"""
    ip, nt = voice(k), geometry(k)["nt"]
    while _g().derive(ip, nf).numberSamples % nt == 0:
        nf += 1
    return nf


def _flagged(ip, nf):
    from gnuspeech_b200 import _native as N
    return bool(N.lib().TRMReferenceFlushBug(C.byref(ip), nf))


def oracle(ip, frames):
    """the oracle's result for one utterance: its ring-buffer converter, or its stateless form where the reference's
    drain would append spurious samples (DESIGN section 7 row 2: the defined output is the stateless one)"""
    f = frames.shape[0]
    return O.synthesize(ip, frames, flags=O.SRC_STATELESS if _flagged(ip, f) else 0, want_tube=False)


# ---- the rate table -------------------------------------------------------------------------------------------------

def test_rate_table_hits_its_cases():
    """Each entry derives the oracle's pad, tri, tube rate and sample counts, and the table holds every case it claims:
    ratio exactly 1, tri 65536 from both sides, either side of 1, each tube rate's lowest accepted rate, a wing that takes
    pad + 1 taps, high up-sampling with nt at its cap, and all four tube rates."""
    geo = [geometry(k) for k in range(len(RATES))]
    for k, s in enumerate(geo):
        ip = voice(k)
        for nf in (1, 2, 3, 40, 151):
            d = _g().derive(ip, nf)
            info = O.OracleInfo()
            assert O.lib().oracle_derive(C.byref(O.as_oracle_ip(ip)), nf, C.byref(info)) == 0, describe(k)
            got = (d.padSize, d.timeRegisterIncrement, d.sampleRate, d.numberSamples)
            want = (info.padSize, info.timeRegisterIncrement, info.sampleRate, info.numberSamples)
            assert got == want, "%s, %d frames: libtrm %s, oracle %s" % (describe(k), nf, got, want)
        assert s["tube_rate"] == TUBE_RATES[RATES[k][1]], describe(k)
        assert s["nt"] >= SRC_CHUNK, describe(k)
    print("\n" + "\n".join(describe(k) for k in range(len(RATES))))
    one = [s for s in geo if s["ratio"] == 1.0]
    assert one and all(s["up"] and s["tri"] == 65536 for s in one)
    for k in entries("tri 65536 from below"):
        assert not geo[k]["up"] and geo[k]["tri"] == 65536 and geo[k]["phaseIncrement"] == 65536 and geo[k]["pad"] == 14, describe(k)
    for k in entries("tri 65536 from above"):
        assert geo[k]["up"] and geo[k]["ratio"] > 1.0 and geo[k]["tri"] == 65536, describe(k)
    for k in entries("just below 1"):
        assert (geo[k]["up"], geo[k]["tri"], geo[k]["phaseIncrement"], geo[k]["pad"]) == (False, 65539, 65533, 14), describe(k)
    for k in entries("just above 1"):
        assert geo[k]["up"] and 65400 < geo[k]["tri"] < 65536, describe(k)
    pad_plus_one = [k for k, s in enumerate(geo) if not s["up"] and math.ceil(851968 / s["phaseIncrement"]) == s["pad"] + 1]
    assert set(entries("pad + 1 taps")) <= set(pad_plus_one) and len(set(TUBE_RATES[RATES[k][1]] for k in pad_plus_one)) >= 3
    high = [s for s in geo if s["ratio"] > 9.0]
    assert high and all(s["nt"] == NT_MAX for s in high)
    bounds = entries("bound")
    assert sorted(RATES[k][1] for k in bounds) == sorted(TUBE_RATES)
    for k in bounds:
        assert geo[k]["nt"] == SRC_CHUNK and geo[k]["pad"] == 47, describe(k)


def test_lowest_accepted_rate_is_refused_at_batch_creation():
    """Bisection on outputRate for each tube rate: the bound entry of RATES is the lowest rate TRMBatchCreate accepts,
    and the next integer rate down is refused there with TRM_ERR_PARAM, not later at synthesis.  libtrm checks the
    window with the exact ratio; plan_chunk sizes work items with the rounded 65536 / tri.  Over 600 rates about each
    bound, both give the same answer (the GPU tests below synthesize at every bound)."""
    g = _g()
    from gnuspeech_b200 import _native as N
    for length in TUBE_RATES:
        low = lowest_accepted_rate(length)
        k = next(k for k in entries("bound") if RATES[k][1] == length)
        assert RATES[k][2] == low, "%g cm: lowest accepted rate %d, table %g" % (length, low, RATES[k][2])
        assert accepted(low - 1, length) == N.TRM_ERR_PARAM
        for out_rate in range(low - 300, low + 300):
            ip = g.TRMInputParameters(float(out_rate), length=length)
            d = g.derive(ip, 2)
            fits = int((SRC_ROWS - 3 - 2 * (d.padSize + 1)) * 65536.0 / d.timeRegisterIncrement) >= SRC_CHUNK
            assert (accepted(out_rate, length) is True) == fits, (length, out_rate)


def test_oracle_ring_equals_stateless_at_every_rate():
    """The oracle is a sound judge at every entry: on short tracks its ring-buffer converter and its stateless form
    give the same samples."""
    for k in range(len(RATES)):
        ip = voice(k)
        for nf, seed in ((1, 1), (2, 2), (41, 3)):
            f = _walk(nf, seed=50 + 10 * k + seed)
            assert not _flagged(ip, nf)
            a = O.synthesize(ip, f, want_tube=False)
            b = O.synthesize(ip, f, flags=O.SRC_STATELESS, want_tube=False)
            assert a.numberSamples == b.numberSamples and np.array_equal(a.samples, b.samples), (describe(k), nf)


# ---- the mixed batch ------------------------------------------------------------------------------------------------

_MIXED = {}


def _mixed():
    """One batch with every entry of RATES: a random walk whose output count is not a multiple of nt, a static vowel,
    1-, 2- and 3-frame walks, and the lengths at which the reference's drain would misbehave, where an entry has one
    below 400 frames.  Returns (ips, frames list, labels, oracle results, entry index per utterance); cached."""
    if not _MIXED:
        from gnuspeech_b200 import workloads as W
        ips, frames, labels, groups = [], [], [], []
        for k in range(len(RATES)):
            ip = voice(k)
            utts = [("walk", _walk(_frames_off_nt(151, k), seed=100 + k)), ("vowel", W.static_vowel(_frames_off_nt(40, k), 1)),
                    ("1 frame", _walk(1, seed=200 + k)), ("2 frames", _walk(2, seed=300 + k)), ("3 frames", _walk(3, seed=400 + k))]
            flagged = [nf for nf in range(4, 400) if _flagged(ip, nf)]
            if flagged:
                utts.append(("drain", _walk(flagged[0], seed=500 + k)))
            for name, f in utts:
                ips.append(ip)
                frames.append(f)
                labels.append("%s %s (%d)" % (describe(k), name, f.shape[0]))
                groups.append(k)
        t = time.time()
        refs = [oracle(ip, f) for ip, f in zip(ips, frames)]
        print("\noracle for %d utterances of the mixed batch: %.1f s" % (len(refs), time.time() - t))
        _MIXED.update(ips=ips, frames=frames, labels=labels, refs=refs, groups=groups)
    return _MIXED["ips"], _MIXED["frames"], _MIXED["labels"], _MIXED["refs"], _MIXED["groups"]


def test_mixed_batch_covers_its_cases():
    """Without a GPU: the mixed batch has output counts off nt's grid, utterances the reference's drain would spoil (whose
    numberSamples libtrm gives as the stateless oracle does), and stereo voices."""
    ips, frames, labels, refs, groups = _mixed()
    b = _g().TRMBatch(list(ips), [f.shape[0] for f in frames])
    flags = b.referenceFlushBugFlags
    assert flags.sum() >= 2
    for u in range(len(ips)):
        assert b.numberSamples[u] == refs[u].numberSamples, labels[u]
    for k in range(len(RATES)):
        walk = next(u for u in range(len(ips)) if groups[u] == k)
        assert b.numberSamples[walk] % geometry(k)["nt"] != 0, labels[walk]
    assert sum(ip.channels == 2 for ip in ips) >= 3


def _synth(ips, frames, n_frames, precision):
    g = _g()
    b = g.TRMBatch(list(ips), list(n_frames), precision=precision)
    pcm = np.zeros(max(1, b.layout.total_pcm_samples), np.int16)
    smp = np.zeros(max(1, b.layout.total_out_samples), b.sample_dtype)
    b.synthesize(np.ascontiguousarray(frames), pcm_out=pcm, samples_out=smp, devices=[0])
    return b, pcm, smp


def _check_pcm(b, pcm, u, ip, ref, label):
    """PCM within 1 LSB of the oracle's; in the FP64 modes the maximum within 1e-9 of the oracle's"""
    peak = ref.maximumSampleValue
    ch = 2 if ip.channels == 2 else 1
    p = pcm[b.pcmOffsets[u]:b.pcmOffsets[u] + b.numberSamples[u] * ch].astype(np.int32)
    d = int(np.abs(p - O.pcm16(ip, ref.samples, peak).astype(np.int32)).max()) if peak else int(np.abs(p).max(initial=0))
    assert d <= 1, "%s: PCM off by %d LSB" % (label, d)
    if b.precision != _g().TRM_PRECISION_FP32:
        assert abs(b.maximumSampleValues[u] - peak) <= FP64_TOL * peak, "%s: maximum %.17g, oracle %.17g" % (label, b.maximumSampleValues[u], peak)
    return d


def _check(b, pcm, smp, cases):
    """cases: (utterance of batch b, voice, oracle result, label).  FP64 modes within 1e-9 of the peak, FP32 at least
    80 dB SNR, PCM within 1 LSB, numberSamples exact.  Returns the worst error (FP64) or SNR (FP32)."""
    is64 = b.precision != _g().TRM_PRECISION_FP32
    worst = 0.0 if is64 else np.inf
    for u, ip, ref, label in cases:
        n = b.numberSamples[u]
        assert n == ref.numberSamples, "%s: numberSamples %d, oracle %d" % (label, n, ref.numberSamples)
        y = smp[b.outOffsets[u]:b.outOffsets[u] + n].astype(np.float64)
        peak = ref.maximumSampleValue
        if n == 0 or peak == 0.0:
            assert not y.any() and b.maximumSampleValues[u] == peak, label
            continue
        if is64:
            e = np.abs(y - ref.samples).max() / peak
            assert e <= FP64_TOL, "%s: FP64 error %.3e of peak" % (label, e)
            worst = max(worst, e)
        else:
            snr = O.snr_db(ref.samples, y)
            assert snr >= FP32_SNR_DB, "%s: SNR %.1f dB" % (label, snr)
            worst = min(worst, snr)
        _check_pcm(b, pcm, u, ip, ref, label)
    return worst


def _same_utterance(b1, pcm1, smp1, u1, b0, pcm0, smp0, u0, ch, what):
    """utterance u1 of batch b1 equals utterance u0 of batch b0 bit for bit: samples, PCM, maximum"""
    k = b0.numberSamples[u0]
    assert b1.numberSamples[u1] == k, what
    o1, o0 = b1.outOffsets[u1], b0.outOffsets[u0]
    assert np.array_equal(smp1[o1:o1 + k], smp0[o0:o0 + k], equal_nan=True), what + ": samples differ"
    p1, p0 = b1.pcmOffsets[u1], b0.pcmOffsets[u0]
    assert np.array_equal(pcm1[p1:p1 + k * ch], pcm0[p0:p0 + k * ch]), what + ": PCM differs"
    assert b1.maximumSampleValues[u1] == b0.maximumSampleValues[u0], what + ": maximum differs"


@gpu
@pytest.mark.parametrize("precision", [0, 1, 2])
def test_every_output_rate_against_the_oracle(precision):
    """Every entry in one batch (tiles of different converter signatures in one chunk) against the oracle, and each
    entry synthesized alone gives the same bytes as inside the mixed batch."""
    ips, frames, labels, refs, groups = _mixed()
    nf = [f.shape[0] for f in frames]
    b, pcm, smp = _synth(ips, np.concatenate(frames), nf, precision)
    worst = _check(b, pcm, smp, list(zip(range(len(ips)), ips, refs, labels)))
    print("\nmixed output rates, precision %d: worst %s %.3g" % (precision, "error/peak" if precision != 1 else "SNR dB", worst))
    for k in range(len(RATES)):
        idx = [u for u in range(len(ips)) if groups[u] == k]
        b1, pcm1, smp1 = _synth([ips[u] for u in idx], np.concatenate([frames[u] for u in idx]), [nf[u] for u in idx], precision)
        for j, u in enumerate(idx):
            _same_utterance(b1, pcm1, smp1, j, b, pcm, smp, u, ips[u].channels, labels[u] + " alone vs mixed")


# ---- the time split and output groups -------------------------------------------------------------------------------

@gpu
@pytest.mark.parametrize("precision", [0, 1, 2])
@pytest.mark.parametrize("case", ["ratio 1", "bound"])
def test_time_split_at_ratio_one_and_the_bound(precision, case, monkeypatch):
    """A uniform batch of 530-frame utterances runs the waveguide as two launches: bit-identical to one launch at
    ratio 1 and at the down-sampling bound, and two utterances against the oracle."""
    k = entries(case)[0]
    n, nf = 9, 530
    kw = [dict(), dict(waveform=1), dict(channels=2, balance=-0.3)]
    ips = [_g().TRMInputParameters(RATES[k][2], length=RATES[k][1], **kw[u % 3]) for u in range(n)]
    frames = np.concatenate([_walk(nf, seed=700 + u) for u in range(n)])
    monkeypatch.delenv("TRM_NO_TIME_SPLIT", raising=False)
    b1, pcm1, smp1 = _synth(ips, frames, [nf] * n, precision)
    assert b1.kernelLaunches == 4                      # two waveguide launches + resampler + PCM
    monkeypatch.setenv("TRM_NO_TIME_SPLIT", "1")
    b0, pcm0, smp0 = _synth(ips, frames, [nf] * n, precision)
    assert b0.kernelLaunches == 3
    for u in range(n):
        _same_utterance(b1, pcm1, smp1, u, b0, pcm0, smp0, u, ips[u].channels, "%s utterance %d" % (describe(k), u))
    _check(b1, pcm1, smp1, [(u, ips[u], oracle(ips[u], frames[u * nf:(u + 1) * nf]), "%s utterance %d" % (describe(k), u))
                            for u in (0, 2)])


@gpu
def test_output_groups_at_192k(monkeypatch):
    """72 utterances of about 10 s at 192 kHz are more than 128 M output samples in one chunk, so the resampler and the
    PCM scaling run in output groups.  Their PCM and maxima equal the single pass, and three utterances match the
    oracle."""
    g = _g()
    k = entries("192 kHz")[0]
    n = 72
    n_frames = [2501 + 3 * u for u in range(n)]          # ragged: no time split
    ips = [voice(k) if u % 2 else g.TRMInputParameters(192000.0, length=RATES[k][1]) for u in range(n)]
    frames = np.concatenate([_walk(nf, seed=900 + u) for u, nf in enumerate(n_frames)])
    res = []
    for off in (False, True):
        if off:
            monkeypatch.setenv("TRM_NO_OUT_GROUPS", "1")
        else:
            monkeypatch.delenv("TRM_NO_OUT_GROUPS", raising=False)
        b = g.TRMBatch(ips, n_frames, precision=g.TRM_PRECISION_FP64)
        assert b.layout.out_samples > 128 << 20
        pcm = np.zeros(b.layout.total_pcm_samples, np.int16)
        b.synthesize(frames, pcm_out=pcm, devices=[0])
        res.append((b, pcm))
    (b1, p1), (b0, p0) = res
    assert b0.kernelLaunches == 3 and b1.kernelLaunches in (5, 7, 9), (b0.kernelLaunches, b1.kernelLaunches)
    assert np.array_equal(b1.maximumSampleValues, b0.maximumSampleValues)
    assert np.array_equal(p1, p0)
    at = np.concatenate(([0], np.cumsum(n_frames)))
    for u in (0, 37, n - 1):
        ref = oracle(ips[u], frames[at[u]:at[u + 1]])
        assert b1.numberSamples[u] == ref.numberSamples
        _check_pcm(b1, p1, u, ips[u], ref, "192 kHz utterance %d" % u)


# ---- streams and the pool -------------------------------------------------------------------------------------------

def _pushes(rng, nf, mmax):
    """random push sizes summing to nf, with 1-frame pushes among them"""
    out = []
    while sum(out) < nf:
        m = 1 if rng.random() < 0.3 else int(rng.integers(1, mmax + 1))
        out.append(min(m, nf - sum(out)))
    return out


STREAM_CASES = [(0, "ratio 1"), (3, "just below 1"), (6, "bound"), (7, "pad + 1 taps"), (10, "192 kHz")]


@gpu
@pytest.mark.parametrize("precision", [0, 1, 2])
@pytest.mark.parametrize("k", [c[0] for c in STREAM_CASES], ids=[c[1] for c in STREAM_CASES])
def test_stream_pushes_at_output_rates(precision, k):
    """TRMStream with random push sizes, 1-frame pushes among them: the concatenated pushes equal the one-shot result
    bit for bit."""
    g = _g()
    assert RATES[k][0] == dict(STREAM_CASES)[k]
    rng = np.random.default_rng(31 * k + precision)
    ip = voice(k)
    n = 3
    nf = _frames_off_nt(int(rng.integers(60, 140)), k)
    frames = np.stack([_walk(nf, seed=1000 + 10 * k + u) for u in range(n)])
    b, _, smp = _synth([ip] * n, frames.reshape(-1, 16), [nf] * n, precision)
    pushes = _pushes(rng, nf, 12)
    st = g.TRMStream(n, ip, precision=precision, max_frames_per_push=max(pushes))
    got = [[] for _ in range(n)]
    at = 0
    for j, m in enumerate(pushes):
        out = st.push(frames[:, at:at + m], flush=(j == len(pushes) - 1))
        at += m
        for u in range(n):
            got[u].append(out[u])
    st.free()
    for u in range(n):
        y = np.concatenate(got[u])
        want = smp[b.outOffsets[u]:b.outOffsets[u] + b.numberSamples[u]]
        assert y.shape == want.shape, (describe(k), y.shape, want.shape)
        assert np.array_equal(y, want, equal_nan=True), "%s, pushes %s: %d samples differ" % (describe(k), pushes, int((y != want).sum()))


class _Slot(object):
    """one utterance streamed through a pool: its frames, its one-shot result, and how far its pushes have come"""

    def __init__(self, k, nf, seed, b, u, pcm, smp):
        self.k, self.nf, self.frames = k, nf, _walk(nf, seed)
        self.ip = voice(k)
        self.ch = 2 if self.ip.channels == 2 else 1
        o, p, n = b.outOffsets[u], b.pcmOffsets[u], b.numberSamples[u]
        self.want, self.want_pcm, self.peak = smp[o:o + n], pcm[p:p + n * self.ch], b.maximumSampleValues[u]
        self.sent = self.at = 0

    def take(self, m):
        f = self.frames[self.sent:self.sent + m]
        self.sent += m
        return f

    def got(self, out, pcm):
        """checks one push's output against the one-shot result, where the slot has got to"""
        if pcm:
            p, _ = out
            n = p.shape[0] // self.ch
            assert np.array_equal(p, self.want_pcm[self.at * self.ch:(self.at + n) * self.ch]), "%s: PCM push at %d" % (describe(self.k), self.at)
        else:
            n = out.shape[0]
            assert np.array_equal(out, self.want[self.at:self.at + n], equal_nan=True), "%s: push at %d" % (describe(self.k), self.at)
        self.at += n


def _slots(ks, precision, rng, lo, hi, seed):
    nfs = [_frames_off_nt(int(rng.integers(lo, hi)), k) for k in ks]
    fr = [_walk(nf, seed + j) for j, nf in enumerate(nfs)]
    b, pcm, smp = _synth([voice(k) for k in ks], np.concatenate(fr), nfs, precision)
    return [_Slot(k, nf, seed + j, b, j, pcm, smp) for j, (k, nf) in enumerate(zip(ks, nfs))]


def _advance(pool, live, rng, mmax, pcm):
    """one push of every live slot by a random frame count (1-frame pushes among them), float or PCM; the slots that
    reach their last frame flush and leave `live`"""
    push, flush = {}, set()
    for s, sl in live.items():
        m = min(1 if rng.random() < 0.3 else int(rng.integers(1, mmax + 1)), sl.nf - sl.sent)
        push[s] = sl.take(m)
        if sl.sent == sl.nf:
            flush.add(s)
    out = pool.push_pcm16(push, {s: live[s].peak for s in push}, flush=flush) if pcm else pool.push(push, flush=flush)
    for s, y in out.items():
        live[s].got(y, pcm)
    for s in flush:
        del live[s]


@gpu
@pytest.mark.parametrize("precision", [0, 1, 2])
def test_pool_slots_at_every_output_rate(precision):
    """One TRMStreamPool with a slot at every entry; the slots open at different pushes, and float and PCM pushes
    alternate at random.  Each slot's output equals its one-shot synthesis bit for bit, and its PCM at the utterance's
    maximumSampleValue equals pcm_out."""
    g = _g()
    rng = np.random.default_rng(55 + precision)
    slots = _slots(range(len(RATES)), precision, rng, 30, 90, seed=1200)
    mmax = 7
    pool = g.TRMStreamPool(len(RATES), precision=precision, max_frames_per_push=mmax)
    waiting = list(range(len(RATES)))
    live = {}
    push = 0
    while live or waiting:
        for j in [j for j in waiting if j % 5 <= push]:     # entry j opens at push j % 5
            live[pool.open(slots[j].ip)] = slots[j]
            waiting.remove(j)
        if live:
            _advance(pool, live, rng, mmax, pcm=rng.random() < 0.5)
        push += 1
    pool.free()
    for sl in slots:
        assert sl.at == sl.want.shape[0], "%s: %d of %d samples" % (describe(sl.k), sl.at, sl.want.shape[0])


@gpu
@pytest.mark.parametrize("precision", [0, 1, 2])
def test_pool_snapshot_at_the_bound_and_192k(precision):
    """The bound-ratio slot and the 192 kHz slot are saved mid-utterance and restored into a pool of another capacity
    and push size that holds a ratio-1 slot, so the restore widens its rows to their pad and output capacity.  The
    restored slots (a migration) and the saved ones (left running: a fork) both continue bit for bit."""
    g = _g()
    rng = np.random.default_rng(91 + precision)
    ks = [entries("ratio 1")[0], entries("bound")[0], entries("192 kHz")[0], entries("ratio 1")[0]]
    slots = _slots(ks, precision, rng, 60, 120, seed=1400)
    a = g.TRMStreamPool(6, precision=precision, max_frames_per_push=5)
    live_a = {a.open(sl.ip): sl for sl in slots[:3]}
    for _ in range(4):
        _advance(a, live_a, rng, 5, pcm=rng.random() < 0.5)
    assert len(live_a) == 3
    saved = a.save([s for s, sl in live_a.items() if sl.k != ks[0]])
    bb = g.TRMStreamPool(11, precision=precision, max_frames_per_push=9)
    live_b = {bb.open(slots[3].ip): slots[3]}
    _advance(bb, live_b, rng, 9, pcm=False)
    forks = {}
    for s, blob in saved.items():
        sl = live_a[s]
        twin = _Slot.__new__(_Slot)
        twin.__dict__.update(sl.__dict__)
        forks[blob] = twin
    for blob, s in zip(saved.values(), bb.restore(list(saved.values()))):
        live_b[s] = forks[blob]
    while live_a or live_b:
        if live_a:
            _advance(a, live_a, rng, 5, pcm=rng.random() < 0.5)
        if live_b:
            _advance(bb, live_b, rng, 9, pcm=rng.random() < 0.5)
    a.free()
    bb.free()
    for sl in slots + list(forks.values()):
        assert sl.at == sl.want.shape[0], "%s: %d of %d samples" % (describe(sl.k), sl.at, sl.want.shape[0])
