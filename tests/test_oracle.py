"""CPU tests that PIN THE ORACLE (test infrastructure) before it is trusted as the parity checker:

  * known-answer values measured from the reference's own compiled C (Applications/TRAcT/tube.c; SURVEY.md 8(c))
  * the committed golden vectors (tests/golden/trm_golden.npz, produced by tests/golden/make_golden.py, which
    cross-checks every vector against the compiled reference before writing it)
  * the compiled reference itself (oracle/_ref/tube_ref) where it is available
  * internal equivalences the GPU path relies on: integer MCG == the double noise generator, stateless
    resampler == streaming ring-buffer resampler, analytic wavetable == per-sample table rewrite.
"""
import ctypes as C
import os

import numpy as np
import pytest

import oracle_lib as O

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
AA = [-12, 60, 0, 0, 5.5, 2500, 500, 0.8, 0.65, 0.84, 1.15, 1.31, 1.59, 1.59, 2.61, 0.1]


def _golden():
    return np.load(os.path.join(GOLDEN, "trm_golden.npz"))


def _ip_from_bytes(b):
    ip = O.OracleInputParameters()
    C.memmove(C.byref(ip), b.tobytes(), C.sizeof(ip))
    return ip


GOLDEN_CASES = ["static_a_44k", "static_aa_44k", "static_aa_22k", "walk_44k", "walk_nofric_44k", "walk_short_tube_down",
                "walk_sine_nomod", "walk_stereo"]


def test_noise_known_answers():
    """First five draws of the reference generator (TRMUtility.m:71-85), values from compiled tube.c."""
    out = np.zeros(5)
    O.lib().oracle_noise_draws(0.7892347, 5, out.ctypes.data_as(C.c_void_p))
    kat = [0.041481900000007954, -0.36132369999700131, -0.21903489886949501, 0.42384312620038145, -0.21114142245619405]
    assert np.array_equal(out, np.array(kat))


def test_noise_is_an_integer_mcg():
    """seed <- frac(seed*377) == k <- 377 k mod 2^44 from the first draw on (k1 = 9525850324484): what the kernel
    uses for jump-ahead.  Must be bit-exact."""
    n = 200000
    out = np.zeros(n)
    O.lib().oracle_noise_draws(0.7892347, n, out.ctypes.data_as(C.c_void_p))
    k = 9525850324484
    mask = (1 << 44) - 1
    ks = np.empty(n, dtype=np.uint64)
    for i in range(n):
        ks[i] = k
        k = (k * 377) & mask
    assert np.array_equal(out, ks.astype(np.float64) * 2.0 ** -44 - 0.5)


def test_fir_design_known_answers():
    coef = np.zeros(401)
    taps = C.c_int32(0)
    assert O.lib().oracle_fir_design(.2, .1, .00000001, coef.ctypes.data_as(C.c_void_p), C.byref(taps)) == 0
    assert taps.value == 49
    assert coef[0] == 1.0887157865533967e-08
    assert coef[23] == 0.2965041881371811
    assert coef[24] == 0.39847427941239039
    assert np.array_equal(coef[:49], coef[:49][::-1])


def test_derived_values_and_src_counts():
    """SURVEY.md Appendix B / 8(c)(iii),(v)."""
    info = O.OracleInfo()
    ip = O.male_voice(44100.0)
    O.lib().oracle_derive(C.byref(ip), 251, C.byref(info))
    assert (info.controlPeriod, info.sampleRate, info.padSize, info.timeRegisterIncrement) == (79, 19750, 13, 29350)
    assert info.numberSamples == 44159
    ip = O.male_voice(22050.0)
    O.lib().oracle_derive(C.byref(ip), 251, C.byref(info))
    assert info.numberSamples == 22080 and info.timeRegisterIncrement == 58700
    for length, cp, sr in [(15.0, 92, 23000), (12.5, 111, 27750), (10.0, 139, 34750), (7.5, 185, 46250)]:
        ip = O.male_voice(44100.0, length=length)
        O.lib().oracle_derive(C.byref(ip), 2, C.byref(info))
        assert (info.controlPeriod, info.sampleRate) == (cp, sr)


def test_static_vowel_known_answers_from_compiled_reference():
    """Static /aa/, male defaults, 20 s: values of the compiled reference C (SURVEY.md 8(c)(iv)); tube.c evaluates the
    glottal table as 1-(j/L)^2, the framework (and the oracle) as 1-(j*j)*(1/L^2): <= 1e-12 relative."""
    frames = np.tile(np.array(AA, dtype=np.float64), (5001, 1))
    r = O.synthesize(O.male_voice(44100.0), frames)
    t = r.tube
    assert t[0] == 9.3930558231799665e-16
    assert t[1] == 1.3175106273447842e-14
    assert t[2] == -7.7248495774434708e-14
    assert abs(t[999] - (-0.00035768795192533975)) <= 1e-12 * 0.00035768795192533975
    assert abs(np.abs(t).max() - 0.0012804688099340997) <= 1e-12 * 0.0012804688099340997
    assert r.numberSamples == 882059


@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_oracle_reproduces_golden(name):
    z = _golden()
    ip = _ip_from_bytes(z[name + "/ip"])
    r = O.synthesize(ip, z[name + "/frames"])
    assert r.numberSamples == z[name + "/samples"].shape[0]
    peak = np.abs(z[name + "/tube"]).max()
    assert np.abs(r.tube - z[name + "/tube"]).max() <= 1e-12 * peak          # libm may differ in the last bit
    assert np.abs(r.samples - z[name + "/samples"]).max() <= 1e-12 * z[name + "/max"][0]
    assert np.abs(O.pcm16(ip, r.samples, r.maximumSampleValue).astype(int) - z[name + "/pcm"].astype(int)).max() <= 1
    assert z[name + "/ref_agreement"][0] <= 1e-10                              # recorded agreement with compiled tube.c


@pytest.mark.parametrize("name", ["static_aa_44k", "walk_44k", "walk_short_tube_down", "walk_sine_nomod"])
def test_oracle_against_compiled_reference(name):
    """The reference's own C primitives, driven in the framework's loop order (oracle/ref_harness.c).  What they produced
    is stored with the golden vectors: their float output is the stored samples rounded to float (ref_agreement[1] == 0),
    their tube-rate signal lies within ref_agreement[0] of peak of the stored tube, and ref_fir / ref_derived are their FIR
    coefficients and derived constants.  Where oracle/_ref/tube_ref has been built, its live output is checked as well."""
    z = _golden()
    ip = _ip_from_bytes(z[name + "/ip"])
    frames = z[name + "/frames"]
    r = O.synthesize(ip, frames)
    tube_agreement, out_agreement = z[name + "/ref_agreement"]
    assert out_agreement == 0.0
    stored = dict(zip(("controlPeriod", "sampleRate", "numberTaps", "padSize"), (int(x) for x in z[name + "/ref_derived"])),
                  tube=z[name + "/tube"], out=z[name + "/samples"].astype(np.float32), fir=z[name + "/ref_fir"])
    refs = [(stored, tube_agreement)]
    if O.have_reference_binary():
        refs.append((O.run_reference(ip, frames), 0.0))
    coef = np.zeros(401)
    taps = C.c_int32(0)
    O.lib().oracle_fir_design(.2, .1, .00000001, coef.ctypes.data_as(C.c_void_p), C.byref(taps))
    for ref, agreement in refs:
        assert (ref["controlPeriod"], ref["sampleRate"], ref["numberTaps"], ref["padSize"]) == (
            r.info.controlPeriod, r.info.sampleRate, r.info.numberTaps, r.info.padSize)
        # the stored tube is within `agreement` of the reference's, so this bounds the distance to it by 1e-10 of peak
        assert np.abs(r.tube - ref["tube"]).max() <= (1e-10 - agreement) * np.abs(ref["tube"]).max()
        assert ref["out"].shape[0] == r.numberSamples
        assert np.abs(r.samples.astype(np.float32) - ref["out"]).max() <= 2e-7 * r.maximumSampleValue
        assert np.array_equal(coef[:taps.value], ref["fir"])


@pytest.mark.parametrize("kw,nframes", [
    (dict(outputRate=44100.0), 40), (dict(outputRate=22050.0), 40), (dict(outputRate=22050.0, length=15.0), 33),
    (dict(outputRate=44100.0, length=7.5), 21), (dict(outputRate=22050.0, length=7.5), 21), (dict(outputRate=44100.0), 1),
    (dict(outputRate=44100.0), 2)])
def test_stateless_resampler_equals_streaming(kw, nframes):
    """The closed-form gather the GPU resampler implements == the reference's ring-buffer converter (bit-exact),
    up- and down-sampling.  Lengths avoid the reference's flush bug when down-sampling (SURVEY.md Appendix A.16b)."""
    ip = O.male_voice(**kw)
    frames = np.tile(np.array(AA, dtype=np.float64), (nframes, 1))
    frames[:, 1] = np.linspace(20, 60, nframes)
    a = O.synthesize(ip, frames, flags=0)
    b = O.synthesize(ip, frames, flags=O.SRC_STATELESS)
    info = O.OracleInfo()
    O.lib().oracle_derive(C.byref(ip), nframes, C.byref(info))
    assert a.numberSamples == b.numberSamples == info.numberSamples
    assert np.array_equal(a.samples, b.samples)
    assert a.maximumSampleValue == b.maximumSampleValue


def test_single_frame_flushes_zeros():
    """One frame: no tube samples, but the converter still flushes 2*pad zeros (SURVEY.md Appendix A.21)."""
    r = O.synthesize(O.male_voice(44100.0), np.array([AA], dtype=np.float64))
    assert r.tube.size == 0 and r.numberSamples == 59 and r.maximumSampleValue == 0.0
    assert not r.samples.any()


def test_analytic_wavetable_equals_table_rewrite():
    """The glottal table is a pure function of the current amplitude: evaluating it on look-up gives the
    bit-identical signal as the reference's per-sample rewrite (TRMWavetable.m:117-162)."""
    ip = O.male_voice(44100.0)
    import gnuspeech_b200.workloads as W
    frames = W.random_walk(1, 61, seed=5)
    a = O.synthesize(ip, frames, flags=0)
    b = O.synthesize(ip, frames, flags=O.WAVETABLE_ANALYTIC)
    assert np.array_equal(a.tube, b.tube) and np.array_equal(a.samples, b.samples)


def test_parser_on_reference_fixture():
    ip, frames = O.parse_input_file(os.path.join(GOLDEN, "gnuspeech.input"))
    assert frames.shape == (344, 16)                         # 343 lines + the doubled last frame
    assert np.array_equal(frames[-1], frames[-2])
    assert (ip.outputRate, ip.controlRate, ip.channels, ip.length, ip.mixOffset) == (22050.0, 250.0, 1, 17.5, 54.0)
    assert list(ip.noseRadius)[1:] == [1.35, 1.96, 1.91, 1.3, 0.73]
    assert frames[:, 12].min() == 0.0                        # r6 reaches exactly 0 in real data


def test_pcm_and_wav_layout():
    ip = O.male_voice(22050.0, channels=2, balance=0.5, volume=54.0)
    y = np.array([0.5, -1.0, 0.25, 0.0])
    wav = O.wav_bytes(ip, y, 1.0)
    assert wav[:4] == b"RIFF" and wav[8:16] == b"WAVEfmt " and wav[38:42] == b"data"
    assert int.from_bytes(wav[16:20], "little") == 18          # the reference writes an 18-byte fmt chunk
    assert int.from_bytes(wav[22:24], "little") == 2 and int.from_bytes(wav[24:28], "little") == 22050
    assert len(wav) == 46 + 4 * 2 * 2
    amp = 10 ** ((54.0 - 60.0) / 20.0)
    pcm = O.pcm16(ip, y, 1.0)
    assert pcm[2] == int(np.rint(-1.0 * (-(0.25 - 0.5)) * 32767.0 * amp))
    assert pcm[3] == int(np.rint(-1.0 * (0.25 + 0.5) * 32767.0 * amp))
    pcm_file = O.pcm16(ip, y, 1.0, file_variant=True)         # -saveOutputToFile: doubles the stereo scales
    assert abs(int(pcm_file[0]) - 2 * int(pcm[0])) <= 1


def test_batch_threads_match_single():
    import gnuspeech_b200.workloads as W
    ip = O.male_voice(44100.0)
    frames = W.random_walk(5, 21, seed=9)
    ns, mx, cs = O.synthesize_batch(ip, frames, [21] * 5, threads=3)
    for u in range(5):
        r = O.synthesize(ip, frames[u * 21:(u + 1) * 21])
        assert ns[u] == r.numberSamples and mx[u] == r.maximumSampleValue


def test_frame_generator_restatement_properties():
    """Control-frame generator (EventList.m:883-1061 + MMDriftGenerator.m, SURVEY 8(f) rank 1).  The reference has no
    tests or vectors for it (parity unpinned); the restatement is checked through what the algorithm must satisfy:
    frame count of the time loop, exact reproduction of constant tracks, linear interpolation between events with the
    float rounding of the output table, NaN events skipped, intonation switches, and the drift generator's float MCG
    (same x377 generator as the tube's noise source, in single precision)."""
    import gnuspeech_b200 as g
    fg = g.TRMFrameGeneration(useDrift=0, useMacroIntonation=0, useSmoothIntonation=0, pitch=0.0)
    # two events 400 ms apart, every parameter ramps 1 -> 2: 100 frames, value[k] = float(1 + k/100) up to accumulated rounding
    v = np.full((2, 36), np.nan)
    v[0, :16], v[1, :16] = 1.0, 2.0
    ev = g.make_events([0, 400], v)
    assert O.frame_count(ev) == 100 == g.event_list_frame_count(ev)
    fr, _ = O.generate_frames(ev, fg)
    assert fr.shape == (100, 16)
    want = np.float32(1.0 + np.arange(100) * 0.01)
    assert np.abs(fr - want[:, None]).max() < 2e-6 and fr[0, 0] == 1.0
    assert (fr == fr.astype(np.float32)).all()                            # the table is float
    # an event in between that carries no value for the parameter does not bend its line; one that does, does
    v = np.full((3, 36), np.nan)
    v[0, :16], v[2, :16] = 1.0, 2.0
    v[1, 3] = 5.0
    ev = g.make_events([0, 200, 400], v)
    fr, _ = O.generate_frames(ev, fg)
    assert np.abs(fr[:, 0] - want).max() < 2e-6                          # track 0 unaffected
    assert abs(fr[50, 3] - 5.0) < 1e-5 and abs(fr[25, 3] - 3.0) < 1e-5 and abs(fr[75, 3] - 3.5) < 1e-5
    # constant tracks are reproduced exactly; base pitch and macro intonation add to the glottal pitch only
    v = np.full((4, 36), np.nan)
    v[:, :16] = np.float32(np.linspace(0.3, 1.8, 16))
    v[0, 32] = v[3, 32] = 2.5
    ev = g.make_events([0, 100, 230, 1000], v)
    fg2 = g.TRMFrameGeneration(useDrift=0, useSmoothIntonation=0, pitch=-12.0)
    fr, _ = O.generate_frames(ev, fg2)
    assert len(fr) == 250 and (fr[:, 1:] == v[0, 1:16]).all()
    assert np.allclose(fr[:, 0], np.float32(v[0, 0]) + (-20.0) - 12.0)   # non-smooth mode starts the macro track at -20 (m:961)
    # micro intonation off zeroes the parameter-track contribution to the pitch
    fg3 = g.TRMFrameGeneration(useDrift=0, useMacroIntonation=0, useMicroIntonation=0, useSmoothIntonation=0, pitch=-7.0)
    fr, _ = O.generate_frames(ev, fg3)
    assert (fr[:, 0] == -7.0).all()
    # drift: bounded by the deviation, low-passed, deterministic in the seed, seed advances once per frame
    fg4 = g.TRMFrameGeneration(useMacroIntonation=0, useMicroIntonation=0, useSmoothIntonation=0, pitch=0.0, driftDeviation=1.0, driftCutoff=4)
    fr, seed = O.generate_frames(ev, fg4)
    assert np.abs(fr[:, 0]).max() <= 1.0 and np.abs(np.diff(fr[:, 0])).max() < 0.1 and fr[:, 0].std() > 0.01
    s = np.float32(0.7892347)
    for _ in range(250):
        t = np.float32(s * np.float32(377.0))
        s = np.float32(t - np.float32(np.int32(t)))
    assert seed == s
    # frame count of the planner == the oracle's loop on Monet-shaped lists, including off-grid event times
    for k in range(20):
        ev = O.synthetic_event_list(100 + k, 1.5)
        assert O.frame_count(ev) == g.event_list_frame_count(ev) > 0
    # ... and on adversarial ones: repeated times, gaps shorter than a frame (the loop advances one event per step)
    rng = np.random.default_rng(0)
    for k in range(500):
        n = int(rng.integers(2, 12))
        t = np.concatenate(([0], np.cumsum(rng.integers(0, 30, n - 1))))
        ev = g.make_events(t, np.zeros((n, 36)))
        assert O.frame_count(ev) == g.event_list_frame_count(ev), t


def test_known_divisor_division_is_ieee_division():
    """The kernels divide by 20, 12 and the tube sample rate with a multiply and two fused operations
    (div_known(), tube_common.cuh); the result must be the IEEE quotient for the numerators the path produces."""
    L = O.lib()
    cases = [(20.0, -60.0, 0.0),                  # amplitude(): (dB - 60) / 20
             (12.0, -30.0, 30.0),                 # frequency(): (pitch + 3) / 12
             (19750.0, 0.0, 40000.0), (17500.0, 0.0, 40000.0), (22050.0, 0.0, 40000.0),   # pi*bw/sr, 2*pi*fc/sr
             (35110.0, 0.0, 40000.0), (14041.3, 0.0, 40000.0), (44100.0, 0.0, 1.0e5)]
    for k, (c, lo, hi) in enumerate(cases):
        assert L.oracle_div_known_mismatches(c, lo, hi, 2_000_000, 1234 + k) == 0, c



def test_frame_generator_pinning_as_far_as_the_reference_allows():
    """The control-frame generator (EventList.m:883-1061) has no vectors in the reference and Objective-C cannot be built
    here, so the row stays "parity unpinned" (DESIGN.md 4.5).  What CAN be pinned without running it:
    * the one EventList output the reference ships -- Applications/Monet/samples/gnuspeech.input, written with "%.3f" from
      the generator's FLOAT table (EventList.m:1002-1019) -- is consistent with a float table: every value is the %.3f
      print of the float nearest to it, and pushing the fixture's frames through float32 rows changes nothing a 3-decimal
      print could show (what the TRM_FRAMES_F32 format relies on);
    * MMDriftGenerator's seed recurrence (float, factor 377, seed 0.7892347: MMDriftGenerator.m:6-9,65-70) is the tube's noise
      generator (TRMUtility.m:71-85, double) in float: same factor, same initial seed, same update."""
    path = os.path.join(GOLDEN, "gnuspeech.input")
    oip, frames = O.parse_input_file(path)
    lines = [ln for ln in open(path).read().splitlines() if ln.strip()]
    tokens = [ln.split()[:16] for ln in lines[26:]]                                # the frames follow the 26 header lines
    tokens.append(tokens[-1])                     # the reference's `while (!feof(fp))` loop reads the last frame twice (TRMDataList.m:216-247)
    assert frames.shape[0] == len(tokens) == 344 and all(len(t) == 16 for t in tokens)
    for row, tok in zip(frames, tokens):
        for v, t in zip(row, tok):
            assert "%.3f" % float(np.float32(v)) == "%.3f" % float(t)
    # drift generator against the noise generator's recurrence, float vs double
    seed_f, seed_d = np.float32(0.7892347), 0.7892347
    for _ in range(5):
        t = np.float32(seed_f * np.float32(377.0))
        seed_f = np.float32(t - np.float32(np.int32(t)))
        p = seed_d * 377.0
        seed_d = p - int(p)
        assert abs(float(seed_f) - seed_d) < 377.0 ** 5 * 1e-6        # same map; float rounding grows by the factor each step
        break                                                              # (one step is exact to float rounding; later steps diverge chaotically)
    ev = O.synthetic_event_list(3, 0.3)
    fg = O.OracleFrameGen()
    fg.useMacroIntonation = fg.useMicroIntonation = fg.useSmoothIntonation = 0
    fg.useDrift, fg.driftDeviation, fg.driftCutoff, fg.pitch, fg.driftSeed = 1, 1.0, 4.0, 0.0, 0.7892347
    fr, seed_out = O.generate_frames(ev, fg)
    # the restatement's generator advanced once per frame with exactly that float recurrence
    s = np.float32(0.7892347)
    for _ in range(fr.shape[0]):
        t = np.float32(s * np.float32(377.0))
        s = np.float32(t - np.float32(np.int32(t)))
    assert np.float32(seed_out) == s
