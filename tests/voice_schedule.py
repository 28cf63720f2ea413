"""The CPU oracle with a voice schedule (tests/voice_schedule_oracle.c): the checker of TRMStreamPoolSetVoice.  Test
infrastructure only.  The library is compiled on first use into a temporary directory (removed at exit) with the
oracle's own flags (oracle/Makefile), so neither the oracle nor the tree changes."""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

import oracle_lib as O

HERE = os.path.dirname(os.path.abspath(__file__))
CFLAGS = ["-O2", "-std=gnu99", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-Wall", "-Wno-unused-function"]

_lib = None


def lib():
    global _lib
    if _lib is None:
        d = tempfile.mkdtemp(prefix="trm_voice_schedule_")
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, "libvoice_schedule.so")
        subprocess.run([os.environ.get("CC", "gcc")] + CFLAGS + ["-shared", "-I" + os.path.join(O.ROOT, "oracle"), "-o", so,
                        os.path.join(HERE, "voice_schedule_oracle.c"), "-lm", "-lpthread"], check=True)
        L = C.CDLL(so)
        L.oracle_synthesize_voices.restype = C.c_int
        L.oracle_synthesize_voices.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p,
                                               C.POINTER(C.POINTER(C.c_double)), C.POINTER(O.OracleInfo)]
        _lib = L
    return _lib


def synthesize_voices(voices, from_sample, frames, flags=0):
    """voices[k] from tube-rate sample from_sample[k] on.  Returns what oracle_lib.synthesize returns; raises with the
    return code (-4: bad schedule or rate constants that differ)."""
    frames = np.ascontiguousarray(frames, dtype=np.float64).reshape(-1, 16)
    n = frames.shape[0]
    ips = (O.OracleInputParameters * len(voices))(*[O.as_oracle_ip(v) for v in voices])
    fs = np.ascontiguousarray(from_sample, dtype=np.int64)
    info = O.OracleInfo()
    rc = O.lib().oracle_derive(C.byref(ips[0]), n, C.byref(info))
    if rc != 0:
        raise RuntimeError("oracle_derive rc=%d" % rc)
    tube = np.zeros(max(1, info.tubeSamples))
    out = C.POINTER(C.c_double)()
    rc = lib().oracle_synthesize_voices(ips, len(voices), fs.ctypes.data_as(C.c_void_p), frames.ctypes.data_as(C.c_void_p), n,
                                        flags, tube.ctypes.data_as(C.c_void_p), C.byref(out), C.byref(info))
    if rc != 0:
        raise RuntimeError("oracle_synthesize_voices rc=%d" % rc)
    r = O.OracleResult()
    r.info = info
    r.numberSamples = info.numberSamples
    r.maximumSampleValue = info.maximumSampleValue
    r.samples = np.ctypeslib.as_array(out, (max(info.numberSamples, 1),))[: info.numberSamples].copy()
    O.lib().oracle_free(out)
    r.tube = tube[: info.tubeSamples]
    r.ip = ips[0]
    return r
