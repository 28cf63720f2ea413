"""Every control period the API accepts, and amplitude()'s clamp at the rounding edge.

The control rate sets the control period cp (tube samples per control frame): 1 Hz gives cp 19,794 and 2.6 kHz the
smallest accepted period, 8.  The paths that depend on cp -- the run-by-run interpolation below 16 samples, the jc0 replay
of streams, pool slots and the time split, the push sizes of the pool, the per-interval seeds of the conformance mode's
recurrences -- are compared with the CPU oracle at each period, in the three arithmetic modes.

amplitude() (TRMUtility.m:26-41) computes `dB -= 60; if (dB <= -60) return 0` in double, which gives 0 for every dB up to
2^-48, and about 1e-3 just above it.  Linear interpolation lands in that window whenever a volume track crosses 0 dB; the
tracks of the clamp tests are chosen, by replaying the reference's interpolation, so that it does."""
import time

import numpy as np
import pytest

import oracle_lib as O

gpu = pytest.mark.gpu

FP64_TOL = 1e-9
FP32_SNR_DB = 80.0
TINY = 2.0 ** -48          # amplitude(dB) is 0 for dB <= TINY: dB - 60 rounds to -60 (half an ulp of 60, ties to even)
F32_EDGE = 2.0 ** -19      # the same rounding in float: (float)dB - 60.f is -60 for dB <= F32_EDGE

# (controlRate, outputRate, tube length, control period, tube rate)
RATES = [
    (1.0, 44100.0, 17.5, 19794, 19794),
    (10.0, 44100.0, 17.5, 1979, 19790),
    (20.0, 22050.0, 17.5, 990, 19800),
    (99.5, 44100.0, 17.5, 199, 19800),
    (250.0, 44100.0, 17.5, 79, 19750),
    (333.3, 44100.0, 17.5, 59, 19664),
    (1000.0, 44100.0, 20.0, 17, 17000),
    (1000.0, 22050.0, 10.0, 35, 35000),     # 35 kHz tube rate to 22.05 kHz: down-sampling
    (1250.0, 44100.0, 17.5, 16, 20000),
    (1600.0, 44100.0, 17.5, 12, 19200),
    (2000.0, 44100.0, 17.5, 10, 20000),
    (2500.0, 44100.0, 17.5, 8, 20000),
    (2600.0, 22050.0, 17.5, 8, 20800),
]
STEREO_CP = 199            # the voice at this period is stereo


def _g():
    import gnuspeech_b200 as g
    return g


def _voice(rate, out_rate=44100.0, length=17.5, **kw):
    ip = _g().TRMInputParameters(out_rate, length=length, **kw)
    ip.controlRate = rate
    return ip


def _voice_of(cp):
    r = next(r for r in RATES if r[3] == cp)
    return _voice(r[0], r[1], r[2])


def _frames_not_on_blocks(n, cp):
    """the smallest frame count >= n whose tube length (n - 1) * cp does not end on a 16-sample block (any n when cp is
    a multiple of 16)"""
    while cp % 16 and ((n - 1) * cp) % 16 == 0:
        n += 1
    return n


def _walk(n, rate, seed):
    """random-walk tracks at control rate `rate`: every frame moves as far as the 250 Hz walk moves in 1 / rate seconds,
    so that at the slow rates each interval is a long pitch and volume ramp"""
    from gnuspeech_b200 import workloads as W
    s = max(1, int(round(250.0 / rate)))
    return np.ascontiguousarray(W.random_walk(1, (n - 1) * s + 1, seed=seed)[::s])


def _check(b, pcm, smp, cases, precision):
    """cases: (utterance of batch b, its voice, its oracle result, label).  FP64 modes within 1e-9 of the peak on the
    samples and the maximum, FP32 at least 80 dB SNR, PCM within 1 LSB.  Returns {label: (worst error or SNR, PCM LSB)}."""
    g = _g()
    ns, po, oo, mx = b.numberSamples, b.pcmOffsets, b.outOffsets, b.maximumSampleValues
    is64 = precision != g.TRM_PRECISION_FP32
    worst = {}
    for u, ip, ref, label in cases:
        assert ns[u] == ref.numberSamples, "%s: numberSamples %d, oracle %d" % (label, ns[u], ref.numberSamples)
        e_w, l_w = worst.get(label, (0.0 if is64 else np.inf, 0))
        peak = ref.maximumSampleValue
        ch = 2 if ip.channels == 2 else 1
        y = smp[oo[u]:oo[u] + ns[u]].astype(np.float64)
        p = pcm[po[u]:po[u] + ns[u] * ch].astype(np.int32)
        if ref.numberSamples == 0 or peak == 0.0:
            assert not y.any() and not p.any() and mx[u] == peak, label
            continue
        if is64:
            e = np.abs(y - ref.samples).max() / peak
            assert e <= FP64_TOL, "%s: FP64 error %.3e of peak" % (label, e)
            assert abs(mx[u] - peak) <= FP64_TOL * peak, "%s: maximum %.17g, oracle %.17g" % (label, mx[u], peak)
            e_w = max(e_w, e)
        else:
            snr = O.snr_db(ref.samples, y)
            assert snr >= FP32_SNR_DB, "%s: SNR %.1f dB" % (label, snr)
            e_w = min(e_w, snr)
        d = int(np.abs(p - O.pcm16(ip, ref.samples, peak).astype(np.int32)).max())
        assert d <= 1, "%s: PCM off by %d LSB" % (label, d)
        worst[label] = (e_w, max(l_w, d))
    return worst


def _print_worst(title, precision, worst):
    unit = "error/peak" if precision != _g().TRM_PRECISION_FP32 else "SNR dB"
    print("\n%s, precision %d (worst %s, PCM LSB):" % (title, precision, unit))
    for k, (e, d) in worst.items():
        print("  %-28s %10.3e  %d" % (k, e, d) if unit == "error/peak" else "  %-28s %10.1f  %d" % (k, e, d))


def _synth(ips, frames, n_frames, precision):
    g = _g()
    b = g.TRMBatch(list(ips), list(n_frames), precision=precision)
    pcm = np.zeros(max(1, b.layout.total_pcm_samples), np.int16)
    smp = np.zeros(max(1, b.layout.total_out_samples), b.sample_dtype)
    b.synthesize(np.ascontiguousarray(frames), pcm_out=pcm, samples_out=smp, devices=[0])
    return b, pcm, smp


def _same_utterance(b1, pcm1, smp1, u1, b0, pcm0, smp0, u0, ch, what):
    """utterance u1 of batch b1 equals utterance u0 of batch b0 bit for bit: samples, PCM, maximum"""
    k = b0.numberSamples[u0]
    assert b1.numberSamples[u1] == k, what
    o1, o0 = b1.outOffsets[u1], b0.outOffsets[u0]
    assert np.array_equal(smp1[o1:o1 + k], smp0[o0:o0 + k], equal_nan=True), what + ": samples differ"
    p1, p0 = b1.pcmOffsets[u1], b0.pcmOffsets[u0]
    assert np.array_equal(pcm1[p1:p1 + k * ch], pcm0[p0:p0 + k * ch]), what + ": PCM differs"
    assert b1.maximumSampleValues[u1] == b0.maximumSampleValues[u0], what + ": maximum differs"


# ---- the mixed-rate batch -------------------------------------------------------------------------------------------

_MIXED = {}


def _mixed():
    """One batch with utterances at every control period: random walks, one-frame and two-frame utterances, a 30 s
    static vowel at 1 Hz, one stereo voice.  Returns (ips, frames list, labels, oracle results); the index into RATES
    of each utterance is in _MIXED["groups"]; cached (the oracle is
    one CPU thread)."""
    if not _MIXED:
        from gnuspeech_b200 import workloads as W
        ips, frames, labels, groups = [], [], [], []
        for k, (rate, out_rate, length, cp, _) in enumerate(RATES):
            kw = dict(channels=2, balance=0.3) if cp == STEREO_CP else {}
            seconds = 6.0 if rate < 5 else (3.0 if rate < 50 else 1.0)
            nf = _frames_not_on_blocks(int(seconds * rate) + 1, cp)
            utts = [("walk", _walk(nf, rate, seed=100 + k))]
            if rate == 1.0:
                utts.append(("vowel", W.static_vowel(_frames_not_on_blocks(31, cp), 1)))    # 30 s, constant increment
            if cp in (19794, 17, 16, 8):
                utts += [("1 frame", _walk(1, rate, seed=200 + k)), ("2 frames", _walk(2, rate, seed=300 + k))]
            for name, f in utts:
                ips.append(_voice(rate, out_rate, length, **kw))
                frames.append(f)
                labels.append("%g Hz cp %d %s (%d)" % (rate, cp, name, f.shape[0]))
                groups.append(k)
        t = time.time()
        refs = [O.synthesize(ip, f, want_tube=False) for ip, f in zip(ips, frames)]
        print("\noracle for %d utterances of the mixed batch: %.1f s" % (len(refs), time.time() - t))
        _MIXED.update(ips=ips, frames=frames, labels=labels, refs=refs, groups=groups)
    return _MIXED["ips"], _MIXED["frames"], _MIXED["labels"], _MIXED["refs"]


def test_control_periods_of_the_rates():
    """The periods and tube rates the tests below rely on (TRMTubeModel.m:196-203)."""
    g = _g()
    for rate, out_rate, length, cp, sr in RATES:
        d = g.derive(_voice(rate, out_rate, length), 10)
        assert (d.controlPeriod, d.sampleRate) == (cp, sr), (rate, length)


@gpu
@pytest.mark.parametrize("precision", [0, 1, 2])
def test_every_control_period_against_the_oracle(precision):
    """All periods in one batch (so a CTA holds utterances with different cp) against the oracle, and each period's
    utterances synthesized alone give the same bytes as in the mixed batch."""
    ips, frames, labels, refs = _mixed()
    t = time.time()
    nf = [f.shape[0] for f in frames]
    b, pcm, smp = _synth(ips, np.concatenate(frames), nf, precision)
    worst = _check(b, pcm, smp, list(zip(range(len(ips)), ips, refs, labels)), precision)
    _print_worst("mixed-rate batch", precision, worst)
    for k in range(len(RATES)):
        idx = [u for u in range(len(ips)) if _MIXED["groups"][u] == k]
        b1, pcm1, smp1 = _synth([ips[u] for u in idx], np.concatenate([frames[u] for u in idx]), [nf[u] for u in idx], precision)
        for j, u in enumerate(idx):
            _same_utterance(b1, pcm1, smp1, j, b, pcm, smp, u, ips[u].channels, labels[u] + " alone vs mixed")
    print("GPU part: %.1f s" % (time.time() - t))


@gpu
@pytest.mark.parametrize("precision", [0, 1, 2])
def test_resident_mixed_rate_batch(precision):
    """TRMBatchMakeResident on the mixed-rate batch: after run() (twice), and on a second resident batch after the stages
    launched one at a time, fetch and fetch_utterance give what TRMBatch.synthesize gives, bit for bit."""
    ips, frames, labels, _ = _mixed()
    nf = [f.shape[0] for f in frames]
    allf = np.ascontiguousarray(np.concatenate(frames))
    b, pcm, smp = _synth(ips, allf, nf, precision)
    g = _g()
    br = g.TRMBatch(list(ips), nf, precision=precision)
    n = len(ips)
    kept = []
    for how in ("run twice", "stage by stage"):
        r = br.make_resident(allf)          # a fresh one, in memory of its own while the first is kept: nothing computed yet
        kept.append(r)
        if how == "run twice":
            r.run()
            r.run()
        else:
            for stage in range(3):
                r.run_stage(stage)
        pcm_r = np.zeros_like(pcm)
        smp_r = np.zeros_like(smp)
        mx_r = np.zeros(n, np.float64)
        r.fetch(pcm_out=pcm_r, samples_out=smp_r, maxima=mx_r)
        assert np.array_equal(mx_r, b.maximumSampleValues), how
        for u in range(n):
            ch = ips[u].channels
            k, o, p = b.numberSamples[u], b.outOffsets[u], b.pcmOffsets[u]
            what = "%s, %s" % (labels[u], how)
            assert np.array_equal(smp_r[o:o + k], smp[o:o + k], equal_nan=True), what + ": fetch samples"
            assert np.array_equal(pcm_r[p:p + k * ch], pcm[p:p + k * ch]), what + ": fetch PCM"
            s1, p1, m1 = r.fetch_utterance(u)
            assert np.array_equal(s1, smp[o:o + k], equal_nan=True), what + ": fetch_utterance samples"
            assert np.array_equal(p1, pcm[p:p + k * ch]), what + ": fetch_utterance PCM"
            assert m1 == b.maximumSampleValues[u], what + ": fetch_utterance maximum"
    for r in kept:
        r.free()


# ---- streams and the pool -------------------------------------------------------------------------------------------

def _pushes(rng, nf, mmax):
    """random push sizes summing to nf, with 1-frame pushes among them"""
    out = []
    while sum(out) < nf:
        m = 1 if rng.random() < 0.3 else int(rng.integers(1, mmax + 1))
        out.append(min(m, nf - sum(out)))
    return out


@gpu
@pytest.mark.parametrize("precision", [0, 1, 2])
@pytest.mark.parametrize("cp", [8, 12, 16, 17, 199, 1979])
def test_stream_pushes_at_other_periods(precision, cp):
    """TRMStream at short and long periods, random push sizes: the concatenated pushes equal the one-shot result bit for
    bit (every push that ends inside a control interval makes the next one replay jc0 interpolation adds)."""
    g = _g()
    rng = np.random.default_rng(cp * 3 + precision)
    rate = next(r[0] for r in RATES if r[3] == cp)
    ip = _voice_of(cp)
    n = 3
    nf = _frames_not_on_blocks(int(rng.integers(20, 40)) if cp > 1000 else int(rng.integers(60, 160)), cp)
    frames = np.stack([_walk(nf, rate, seed=400 + 10 * cp + u) for u in range(n)])
    b, _, smp = _synth([ip] * n, frames.reshape(-1, 16), [nf] * n, precision)
    pushes = _pushes(rng, nf, 12)
    st = g.TRMStream(n, ip, precision=precision, max_frames_per_push=max(pushes))
    got = [[] for _ in range(n)]
    at = 0
    for k, m in enumerate(pushes):
        out = st.push(frames[:, at:at + m], flush=(k == len(pushes) - 1))
        at += m
        for u in range(n):
            got[u].append(out[u])
    st.free()
    for u in range(n):
        y = np.concatenate(got[u])
        want = smp[b.outOffsets[u]:b.outOffsets[u] + b.numberSamples[u]]
        assert y.shape == want.shape, (u, y.shape, want.shape)
        assert np.array_equal(y, want, equal_nan=True), "stream %d, pushes %s: %d samples differ" % (u, pushes, int((y != want).sum()))


@gpu
@pytest.mark.parametrize("precision", [0, 1, 2])
def test_pool_slots_at_different_control_rates(precision):
    """TRMStreamPool slots at 8 different periods, advanced together by every push.  The long-period slots open after the
    first push, so the pool widens its rows while the other slots carry history.  Each slot equals its one-shot
    TRMBatch synthesis bit for bit."""
    g = _g()
    rng = np.random.default_rng(77 + precision)
    cps = [8, 12, 17, 35, 79, 199, 1979, 19794]
    ips = [_voice_of(cp) for cp in cps]
    rates = [next(r[0] for r in RATES if r[3] == cp) for cp in cps]
    nfs = [_frames_not_on_blocks(int(rng.integers(30, 80)) if cp < 1000 else int(rng.integers(4, 12)), cp) for cp in cps]
    frames = [_walk(nf, rate, seed=600 + k) for k, (nf, rate) in enumerate(zip(nfs, rates))]
    b, _, smp = _synth(ips, np.concatenate(frames), nfs, precision)
    want = [smp[b.outOffsets[u]:b.outOffsets[u] + b.numberSamples[u]] for u in range(len(cps))]
    mmax = 6
    pool = g.TRMStreamPool(len(cps), precision=precision, max_frames_per_push=mmax)
    slots, sent, got = {}, [0] * len(cps), [[] for _ in cps]
    later = [k for k in range(len(cps)) if cps[k] >= 1000]
    for k in range(len(cps)):
        if k not in later:
            slots[pool.open(ips[k])] = k
    while slots:
        push, flush = {}, set()
        for s, k in slots.items():
            m = min(1 if rng.random() < 0.3 else int(rng.integers(1, mmax + 1)), nfs[k] - sent[k])
            push[s] = frames[k][sent[k]:sent[k] + m]
            sent[k] += m
            if sent[k] == nfs[k]:
                flush.add(s)
        out = pool.push(push, flush=flush)
        for s, y in out.items():
            got[slots[s]].append(y)
        for s in flush:
            del slots[s]
        for k in later:
            slots[pool.open(ips[k])] = k
        later = []
    pool.free()
    for k in range(len(cps)):
        y = np.concatenate(got[k])
        assert y.shape == want[k].shape, (cps[k], y.shape, want[k].shape)
        assert np.array_equal(y, want[k], equal_nan=True), "slot at cp %d: %d samples differ" % (cps[k], int((y != want[k]).sum()))


# ---- the time split -------------------------------------------------------------------------------------------------

@gpu
@pytest.mark.parametrize("precision", [0, 1, 2])
@pytest.mark.parametrize("cp", [10, 990])
def test_time_split_at_other_periods(precision, cp, monkeypatch):
    """A uniform batch of 530-frame utterances runs the waveguide as two launches; the second starts inside a control
    interval (jc0 2 at cp 10, 982 at cp 990).  Bit-identical to one launch; two utterances against the oracle."""
    rate, out_rate, length = next(r[:3] for r in RATES if r[3] == cp)
    voices = [dict(), dict(waveform=1), dict(usesModulation=0, breathiness=3.0), dict(channels=2, balance=-0.3), dict(lossFactor=1.2)]
    n, nf = 9, 530
    ips = [_voice(rate, out_rate, length, **voices[u % len(voices)]) for u in range(n)]
    frames = np.concatenate([_walk(nf, rate, seed=700 + u) for u in range(n)])
    monkeypatch.delenv("TRM_NO_TIME_SPLIT", raising=False)
    b1, pcm1, smp1 = _synth(ips, frames, [nf] * n, precision)
    assert b1.kernelLaunches == 4                      # two waveguide launches + resampler + PCM
    monkeypatch.setenv("TRM_NO_TIME_SPLIT", "1")
    b0, pcm0, smp0 = _synth(ips, frames, [nf] * n, precision)
    assert b0.kernelLaunches == 3
    for u in range(n):
        _same_utterance(b1, pcm1, smp1, u, b0, pcm0, smp0, u, ips[u].channels, "utterance %d" % u)
    cases = [(u, ips[u], O.synthesize(ips[u], frames[u * nf:(u + 1) * nf], want_tube=False), "cp %d utterance %d" % (cp, u))
             for u in (0, 3)]
    _print_worst("time split at cp %d" % cp, precision, _check(b1, pcm1, smp1, cases, precision))


# ---- amplitude()'s clamp window -------------------------------------------------------------------------------------

def interpolated(a, b, cp):
    """the values one parameter takes over the control interval from frame value a to frame value b, as the reference
    computes them (TRMTubeModel.m:611-688): p = a; d = (b - a) / cp; one p += d after each sample"""
    p, d = a, (b - a) / cp
    out = np.empty(cp)
    for i in range(cp):
        out[i] = p
        p += d
    return out


def crossing_pairs(cp, lo, hi):
    """(a, b) frame pairs, a in -0.1 .. -6 dB, b in 0.1 .. 30 dB (decimal doubles and their float roundings, as Monet's
    frames carry), whose interpolation at period cp takes a value in (lo, hi]"""
    a, b = [x.ravel() for x in np.meshgrid(-np.arange(1, 61) / 10.0, np.arange(1, 301) / 10.0)]
    a = np.concatenate([a, a.astype(np.float32).astype(np.float64)])
    b = np.concatenate([b, b.astype(np.float32).astype(np.float64)])
    p, d = a.copy(), (b - a) / cp
    hit = np.zeros(a.shape, bool)
    for _ in range(cp):
        hit |= (p > lo) & (p <= hi)
        p = p + d
    return [(float(x), float(y)) for x, y in zip(a[hit], b[hit])]


WINDOWS = {"conformance": (0.0, TINY), "fast": (TINY, np.nextafter(F32_EDGE, 0.0))}
CLAMP_COLS = {1: "glottal", 2: "aspiration", 3: "frication"}


def clamp_track(cp, col, seed, n_each=6):
    """A static /aa/ whose volume `col` crosses 0 dB n_each times through each window, between stretches at its usual
    level (60 dB glottal, 40 dB aspiration and frication with the frication tap inside the tube)."""
    from gnuspeech_b200 import workloads as W
    rng = np.random.default_rng(seed)
    level = 60.0 if col == 1 else 40.0
    vals = []
    for lo, hi in WINDOWS.values():
        pairs = crossing_pairs(cp, lo, hi)
        for i in rng.choice(len(pairs), n_each, replace=False):
            vals += [pairs[i][0], pairs[i][1], level]
    fr = W.static_vowel(len(vals) + 2, 1)
    fr[:, col] = level
    fr[1:1 + len(vals), col] = vals
    if col == 3:
        fr[:, 4] = 5.3
    return fr


def _clamp_cases():
    out = []
    for cp, rate, length in ((79, 250.0, 17.5), (17, 1000.0, 20.0)):
        for col in CLAMP_COLS:
            out.append((cp, col, _voice(rate, 44100.0, length), clamp_track(cp, col, seed=cp * 10 + col)))
    return out


def test_clamp_tracks_hit_both_windows():
    """Every clamp track really puts interpolated values in (0, 2^-48] and in (2^-48, 2^-19), so the GPU test below keeps
    exercising both windows."""
    for cp, col, ip, fr in _clamp_cases():
        v = np.concatenate([interpolated(fr[i, col], fr[i + 1, col], cp) for i in range(fr.shape[0] - 1)])
        for name, (lo, hi) in WINDOWS.items():
            hits = int(((v > lo) & (v <= hi)).sum())
            assert hits >= 6, "cp %d %s: %d values in the %s window" % (cp, CLAMP_COLS[col], hits, name)


def test_oracle_amplitude_at_the_clamp_edge():
    """The oracle's amplitude() is the reference's: 0 up to 2^-48 (ties to -60), 1e-3 just above, 0 for -0 and below."""
    amp = O.lib().oracle_amplitude
    for db in (TINY, 0.0, -0.0, -1e-300, -5.0, 5e-324, TINY / 2):
        assert amp(db) == 0.0, db
    for db in (np.nextafter(TINY, 1.0), 2 * TINY, 1e-10, F32_EDGE, 1e-6):
        assert amp(db) == pytest.approx(10.0 ** ((db - 60.0) / 20.0), rel=1e-14), db
        assert amp(db) == pytest.approx(1e-3, rel=1e-6), db


@gpu
@pytest.mark.parametrize("precision", [0, 1, 2])
def test_clamp_window_against_the_oracle(precision):
    """Glottal, aspiration and frication volume crossing 0 dB through both windows, at cp 79 and 17: every mode within its
    tolerance of the oracle.  A clamp decided as `dB <= 0` (or on the float parameter) gives 1e-3 where the reference
    gives 0 (or the reverse): a 60 dB step on one sample."""
    cases = _clamp_cases()
    ips = [c[2] for c in cases]
    frames = [c[3] for c in cases]
    labels = ["cp %d %s" % (c[0], CLAMP_COLS[c[1]]) for c in cases]
    refs = [O.synthesize(ip, f, want_tube=False) for ip, f in zip(ips, frames)]
    b, pcm, smp = _synth(ips, np.concatenate(frames), [f.shape[0] for f in frames], precision)
    _print_worst("clamp window", precision, _check(b, pcm, smp, list(zip(range(len(ips)), ips, refs, labels)), precision))


def push_starts(pushes, cp):
    """(control interval, jc0) at which each push after the first starts: TRMStream synthesizes the whole 16-sample blocks
    of the tube samples that the frames seen so far define, (frames - 1) * cp, and the next push replays the first jc0
    interpolation adds of the interval it starts in"""
    seen, done, out = 0, 0, []
    for m in pushes[:-1]:
        seen += m
        if seen >= 2:
            done = (seen - 1) * cp // 16 * 16
        out.append((done // cp, done % cp))
    return out


def _boundary_crossings(cp, fr, col, pushes):
    """per window: the pushes that start inside an interval whose interpolation hits that window"""
    starts = [(f, j) for f, j in push_starts(pushes, cp) if j > 0]
    found = {}
    for name, (lo, hi) in WINDOWS.items():
        found[name] = [(f, j) for f, j in starts
                       if f + 1 < fr.shape[0] and ((interpolated(fr[f, col], fr[f + 1, col], cp) > lo) &
                                                   (interpolated(fr[f, col], fr[f + 1, col], cp) <= hi)).any()]
    return found


def test_push_boundaries_fall_inside_the_crossing_intervals():
    """With the 1-frame pushes of the GPU test below, pushes start inside the crossing intervals of every clamp track,
    for both windows, so the jc0 replay runs the interpolation through the window."""
    for cp, col, _, fr in _clamp_cases():
        pushes = [1] * fr.shape[0]
        for name, hits in _boundary_crossings(cp, fr, col, pushes).items():
            assert len(hits) >= 4, "cp %d %s, %s window: pushes start in %d crossing intervals" % (cp, CLAMP_COLS[col], name, len(hits))


@gpu
@pytest.mark.parametrize("precision", [0, 1, 2])
@pytest.mark.parametrize("cp", [79, 17])
def test_clamp_window_across_push_boundaries(precision, cp):
    """The clamp tracks streamed one frame per push: pushes start inside the crossing intervals (checked above) and
    replay the interpolation adds through the window.  Equal to the one-shot result bit for bit."""
    g = _g()
    cases = [c for c in _clamp_cases() if c[0] == cp]
    ip = cases[0][2]
    frames = np.stack([c[3] for c in cases])
    n, nf = frames.shape[:2]
    b, _, smp = _synth([ip] * n, frames.reshape(-1, 16), [nf] * n, precision)
    pushes = [1] * nf
    st = g.TRMStream(n, ip, precision=precision, max_frames_per_push=1)
    got = [[] for _ in range(n)]
    at = 0
    for k, m in enumerate(pushes):
        out = st.push(frames[:, at:at + m], flush=(k == len(pushes) - 1))
        at += m
        for u in range(n):
            got[u].append(out[u])
    st.free()
    for u in range(n):
        y = np.concatenate(got[u])
        want = smp[b.outOffsets[u]:b.outOffsets[u] + b.numberSamples[u]]
        assert np.array_equal(y, want, equal_nan=True), "%s: %d samples differ" % (CLAMP_COLS[cases[u][1]], int((y != want).sum()))
