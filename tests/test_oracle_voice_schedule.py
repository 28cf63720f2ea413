"""CPU tests of the oracle with a voice schedule (tests/voice_schedule_oracle.c, oracle_synthesize_voices), the checker
of TRMStreamPoolSetVoice: a stream whose voice changes while it plays, every state variable carried across the change."""
import numpy as np
import pytest

import oracle_lib as O
import voice_schedule as V

AA = np.array([-12, 60, 0, 0, 5.5, 2500, 500, 0.8, 0.65, 0.84, 1.15, 1.31, 1.59, 1.59, 2.61, 0.1])


def _frames(n, seed):
    """A vowel with wandering pitch, volumes and radii, and some frication."""
    rng = np.random.default_rng(seed)
    f = np.tile(AA, (n, 1))
    f[:, 0] += np.cumsum(rng.normal(0, 0.4, n))
    f[:, 2] = np.clip(np.cumsum(rng.normal(0, 1, n)), 0, 10)
    f[:, 3] = np.clip(np.cumsum(rng.normal(0, 2, n)), 0, 24)
    f[:, 7:15] = np.clip(f[:, 7:15] + np.cumsum(rng.normal(0, 0.03, (n, 8)), axis=0), 0.05, 3.0)
    return f


def test_one_voice_schedule_is_oracle_synthesize():
    ip = O.male_voice()
    fr = _frames(60, 1)
    for flags in (0, O.WAVETABLE_ANALYTIC, O.SRC_STATELESS):
        a = O.synthesize(ip, fr, flags)
        b = V.synthesize_voices([ip], [0], fr, flags)
        assert np.array_equal(a.tube, b.tube) and np.array_equal(a.samples, b.samples)
        assert a.maximumSampleValue == b.maximumSampleValue and a.info.finalNoiseSeed == b.info.finalNoiseSeed


@pytest.mark.parametrize("at", [0, 1, 2222, 4000])
def test_same_voice_twice_changes_nothing(at):
    ip = O.male_voice()
    fr = _frames(60, 2)
    a = O.synthesize(ip, fr)
    b = V.synthesize_voices([ip, O.male_voice()], [0, at], fr)
    assert np.array_equal(a.tube, b.tube) and np.array_equal(a.samples, b.samples)


def test_change_takes_effect_at_its_sample():
    """Samples before from_sample are the first voice's; from there on they differ."""
    v1, v2 = O.male_voice(), O.male_voice(breathiness=4.0, lossFactor=1.5, throatVol=20.0)
    fr = _frames(60, 3)
    a = O.synthesize(v1, fr)
    at = 2001
    b = V.synthesize_voices([v1, v2], [0, at], fr)
    assert np.array_equal(a.tube[:at], b.tube[:at])
    assert b.tube[at] != a.tube[at]


@pytest.mark.parametrize("change", [dict(tp=30.0, tnMax=40.0), dict(tnMin=8.0), dict(waveform=1), dict(waveform=0)])
def test_analytic_and_rewriting_tables_agree_across_a_change(change):
    w1 = dict(waveform=1) if change.get("waveform") == 0 else {}
    v1, v2 = O.male_voice(**w1), O.male_voice(**change)
    fr = _frames(60, 4)
    a = V.synthesize_voices([v1, v2, v1], [0, 1501, 3000], fr, 0)
    b = V.synthesize_voices([v1, v2, v1], [0, 1501, 3000], fr, O.WAVETABLE_ANALYTIC)
    assert np.array_equal(a.tube, b.tube)


@pytest.mark.parametrize("change", [dict(length=15.0), dict(temperature=35.0), dict(outputRate=22050.0),
                                    dict(controlRate=200.0), dict(channels=2)])
def test_rate_constants_must_stay(change):
    fr = _frames(20, 5)
    with pytest.raises(RuntimeError, match="rc=-4"):
        V.synthesize_voices([O.male_voice(), O.male_voice(**change)], [0, 100], fr)


def test_length_that_rounds_to_the_same_period_is_accepted():
    fr = _frames(20, 6)
    v1, v2 = O.male_voice(), O.male_voice(length=17.5001)
    assert V.synthesize_voices([v1, v2], [0, 100], fr).numberSamples == O.synthesize(v1, fr).numberSamples


def test_bad_schedule():
    fr = _frames(20, 7)
    v = O.male_voice()
    for sched in ([5, 10], [0, 10, 9]):
        with pytest.raises(RuntimeError, match="rc=-4"):
            V.synthesize_voices([v] * len(sched), sched, fr)
