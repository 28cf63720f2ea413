"""TRMStream's outward behaviour beyond the samples: the capacity it reports, its refusals (codes and messages), a flush
before any frame, and a push whose samples are not wanted (samples_out = NULL).  The values were recorded from the
implementation that advanced the streams with its own lockstep engine (B200), before TRMStream became a lockstep use of
the stream pool; the samples themselves are checked against the one-shot path by test_gpu_stream.py."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _g():
    import gnuspeech_b200 as g
    return g


def _voice(name):
    g = _g()
    if name == "male":
        return g.TRMInputParameters(44100.0)
    if name == "female":
        ip = g.MMSynthesisParameters("Female").inputParameters()
        ip.channels = 1
        return ip
    return g.TRMInputParameters(22050.0, length=10.0)      # 10 cm tract at 22.05 kHz: the converter down-samples


CAPACITY = {
    ("male", 1): 640, ("male", 8): 1888, ("male", 125): 22528,
    ("female", 1): 608, ("female", 8): 1856, ("female", 125): 22496,
    ("short", 1): 320, ("short", 8): 928, ("short", 125): 11264,
}


@pytest.mark.parametrize("precision", [0, 1, 2])
@pytest.mark.parametrize("voice,max_frames", sorted(CAPACITY))
def test_capacity(voice, max_frames, precision):
    g = _g()
    st = g.TRMStream(2, _voice(voice), precision=precision, max_frames_per_push=max_frames)
    got = st.capacity
    st.free()
    assert got == CAPACITY[(voice, max_frames)], (voice, max_frames, precision, got)


def _push(st, frames, m, flush, out):
    """TRMStreamPush through the C ABI: (return code, message, n_samples)."""
    from gnuspeech_b200 import _native as N
    k = C.c_int64(-1)
    fp = frames.ctypes.data_as(C.c_void_p) if frames is not None else None
    op = out.ctypes.data_as(C.c_void_p) if out is not None else None
    rc = N.lib().TRMStreamPush(st._h if st is not None else None, fp, m, flush, op, C.byref(k))
    return rc, N.lib().TRMLastErrorMessage().decode(), k.value


def _one_shot(ip, frames, prec):
    g = _g()
    n, nf = frames.shape[0], frames.shape[1]
    b = g.TRMBatch(ip, [nf] * n, precision=prec)
    smp = np.zeros(b.layout.total_out_samples, b.sample_dtype)
    b.synthesize(frames.reshape(n * nf, 16), samples_out=smp, devices=[0])
    return [smp[b.outOffsets[u]:b.outOffsets[u] + b.numberSamples[u]] for u in range(n)]


def test_refusals():
    """m = -1 and m = max + 1 are refused and change nothing (the pushes that follow still give the one-shot result); a
    push after the flush is refused; a NULL stream too."""
    g = _g()
    from gnuspeech_b200 import _native as N
    from gnuspeech_b200 import workloads as W
    ip = _voice("male")
    n, nf, mx = 2, 24, 8
    frames = W.random_walk(n, nf, seed=31).reshape(n, nf, 16)
    want = _one_shot(ip, frames, 0)
    st = g.TRMStream(n, ip, precision=0, max_frames_per_push=mx)
    more = "CUDA: trm_cuda_stream_push: more frames than the stream was created for"
    big = np.zeros((n, mx + 1, 16))
    assert _push(st, big, -1, 0, st._buf) == (N.TRM_ERR_CUDA, more, 0)
    got = []
    for at in range(0, nf, mx):
        assert _push(st, big, mx + 1, 0, st._buf) == (N.TRM_ERR_CUDA, more, 0)
        got.append(st.push(frames[:, at:at + mx], flush=(at + mx >= nf)))
    y = np.concatenate(got, axis=1)
    for u in range(n):
        assert np.array_equal(y[u], want[u]), u
    flushed = "CUDA: trm_cuda_stream_push: the streams were flushed"
    assert _push(st, frames[:, :1].copy(), 1, 0, st._buf) == (N.TRM_ERR_CUDA, flushed, 0)
    assert _push(st, None, 0, 1, st._buf) == (N.TRM_ERR_CUDA, flushed, 0)
    st.free()
    assert _push(None, None, 0, 0, None)[:2] == (N.TRM_ERR_PARAM, "null stream")


@pytest.mark.parametrize("precision", [0, 1])
def test_flush_before_any_frame(precision):
    """A flush with no frame ever pushed returns no samples and ends the streams."""
    g = _g()
    from gnuspeech_b200 import _native as N
    st = g.TRMStream(3, _voice("male"), precision=precision, max_frames_per_push=4)
    rc, _, k = _push(st, None, 0, 1, st._buf)
    assert (rc, k) == (N.TRM_OK, 0)
    assert _push(st, None, 0, 0, st._buf)[:2] == (N.TRM_ERR_CUDA, "CUDA: trm_cuda_stream_push: the streams were flushed")
    st.free()


@pytest.mark.parametrize("precision", [0, 1])
def test_push_without_samples_out(precision):
    """A push with samples_out = NULL advances the streams and reports its count; the samples it does not copy are
    the one-shot result's first ones, and the pushes after it continue that result bit for bit."""
    g = _g()
    from gnuspeech_b200 import _native as N
    from gnuspeech_b200 import workloads as W
    ip = _voice("female")
    n, nf = 3, 41
    frames = W.random_walk(n, nf, seed=37).reshape(n, nf, 16)
    want = _one_shot(ip, frames, precision)
    st = g.TRMStream(n, ip, precision=precision, max_frames_per_push=8)
    rc, _, k0 = _push(st, np.ascontiguousarray(frames[:, :8]), 8, 0, None)
    assert rc == N.TRM_OK and k0 > 0
    got = [st.push(frames[:, at:at + 8], flush=(at + 8 >= nf)) for at in range(8, nf, 8)]
    st.free()
    y = np.concatenate(got, axis=1)
    for u in range(n):
        assert np.array_equal(y[u], want[u][k0:]), u
