"""Streaming synthesis (TRMStream; SURVEY 8(f) rank 3, TRAcT's mode of use): control frames pushed in pieces, un-normalised
samples returned as they become computable, all recurrence state carried on the device.  The contract: whatever the
push sizes, the concatenated output is bit-identical to synthesizing the whole utterance at once."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _g():
    import gnuspeech_b200 as g
    return g


def _one_shot(ip, frames, n, nf, prec):
    g = _g()
    b = g.TRMBatch(ip, [nf] * n, precision=prec)
    smp = np.zeros(b.layout.total_out_samples, b.sample_dtype)
    b.synthesize(frames.reshape(n * nf, 16), samples_out=smp, devices=[0])
    ns, oo = b.numberSamples, b.outOffsets
    return [smp[oo[u]:oo[u] + ns[u]] for u in range(n)]


@pytest.mark.parametrize("precision", [0, 1])
@pytest.mark.parametrize("pushes", [[13, 1, 1, 7, 40, 3, 60], [125], [2] * 62 + [1]])
def test_pushes_concatenate_to_the_one_shot_result(precision, pushes):
    g = _g()
    from gnuspeech_b200 import workloads as W
    n, nf = 5, sum(pushes)
    ip = g.TRMInputParameters(44100.0)
    frames = W.random_walk(n, nf, seed=17).reshape(n, nf, 16)
    want = _one_shot(ip, frames, n, nf, precision)
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
        assert y.shape == want[u].shape, (u, y.shape, want[u].shape)
        assert np.array_equal(y, want[u]), "stream %d: %d samples differ, first at %d" % (
            u, int((y != want[u]).sum()), int(np.nonzero(y != want[u])[0][0]))


def test_stream_latency_and_other_voice():
    """A push returns everything computable from the frames so far (at most one 16-sample waveguide block and the
    converter's right wing are held back); a shorter tract (female voice, 23 kHz tube rate) streams the same way."""
    g = _g()
    from gnuspeech_b200 import workloads as W
    ip = g.MMSynthesisParameters("Female").inputParameters()
    ip.channels = 1
    n, nf = 3, 41
    frames = W.random_walk(n, nf, seed=23).reshape(n, nf, 16)
    want = _one_shot(ip, frames, n, nf, g.TRM_PRECISION_FP64)
    st = g.TRMStream(n, ip, precision=g.TRM_PRECISION_FP64, max_frames_per_push=8)
    got, produced = [], 0
    cp = g.derive(ip, nf).controlPeriod
    for at in range(0, nf, 8):
        m = min(8, nf - at)
        out = st.push(frames[:, at:at + m], flush=(at + m == nf))
        produced += out.shape[1]
        got.append(out)
        if at + m < nf:
            tube_so_far = (at + m - 1) * cp
            assert produced >= int((tube_so_far - 16) * 44100.0 / (250.0 * cp)) - 2      # within one block of real time
    st.free()
    y = np.concatenate(got, axis=1)
    for u in range(n):
        assert np.array_equal(y[u], want[u]), u


@pytest.mark.parametrize("precision", [0, 1])
def test_down_sampling_voice_streams_too(precision):
    """A 10 cm tract at 22.05 kHz output: the tube runs at 35 kHz and the converter down-samples (phase-walking taps, 22
    pad samples per wing).  Same contract: the pushes concatenate to the one-shot result, bit for bit."""
    g = _g()
    from gnuspeech_b200 import workloads as W
    ip = g.TRMInputParameters(22050.0, length=10.0)
    pushes = [9, 1, 2, 30, 5, 17]
    n, nf = 3, sum(pushes)
    frames = W.random_walk(n, nf, seed=29).reshape(n, nf, 16)
    want = _one_shot(ip, frames, n, nf, precision)
    st = g.TRMStream(n, ip, precision=precision, max_frames_per_push=max(pushes))
    got, at = [], 0
    for k, m in enumerate(pushes):
        got.append(st.push(frames[:, at:at + m], flush=(k == len(pushes) - 1)))
        at += m
    st.free()
    y = np.concatenate(got, axis=1)
    for u in range(n):
        assert y[u].shape == want[u].shape, (u, y[u].shape, want[u].shape)
        assert np.array_equal(y[u], want[u]), "stream %d: %d samples differ, first at %d" % (
            u, int((y[u] != want[u]).sum()), int(np.nonzero(y[u] != want[u])[0][0]))


import oracle_lib as O  # noqa: E402


@pytest.mark.parametrize("case", ["walk_44k", "walk_short_tube_down"])
def test_stream_against_the_reference_float_stream(case):
    """TRAcT's mode of use, checked against the reference itself: Applications/TRAcT/tube.c's converter (dataFill /
    dataEmpty, tube.c:2348-2521) emits the un-normalised FLOAT stream TRAcT plays (tube.c:1096-1191).  The golden vectors
    hold that stream: tests/golden/make_golden.py ran the compiled tube.c on these frames and recorded that the stored
    samples, rounded to float, were identical to its output (ref_agreement[1] == 0).  TRMStream, fed the same frames in
    small pushes, must return that stream -- to the float precision tube.c emits (2e-7 of peak, as tests/test_oracle.py
    uses for the same comparison)."""
    import os
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
    st = g.TRMStream(1, ip, precision=g.TRM_PRECISION_FP64, max_frames_per_push=16)
    parts, at = [], 0
    for m in ([5, 1, 16, 3] * nf)[:nf]:
        m = min(m, nf - at)
        if m <= 0:
            break
        parts.append(st.push(frames[None, at:at + m], flush=(at + m >= nf))[0])
        at += m
    st.free()
    y = np.concatenate(parts)
    assert y.shape[0] == ref_out.shape[0]
    peak = float(np.abs(ref_out).max())
    assert np.abs(y.astype(np.float32) - ref_out).max() <= 2e-7 * peak
