"""Generates tests/golden/trm_golden.npz: small input/output vectors for the TRM hot path.

Run in the build container (where /root/reference is mounted):   python tests/golden/make_golden.py

Every vector is produced by the CPU oracle (oracle/trm_oracle.c) AND, for the tube-rate signal, checked here
against the REFERENCE'S OWN compiled C (Applications/TRAcT/tube.c via oracle/_ref/tube_ref) before it is
written; the agreement (max relative difference) is stored next to each vector, together with the reference's FIR
coefficients (ref_fir) and its controlPeriod, sampleRate, numberTaps and padSize (ref_derived).  The reference ships no
golden audio of its own (SURVEY.md section 4), so these files are the pinned contract.

ref_fir and ref_derived of static_aa_44k, walk_44k, walk_short_tube_down and walk_sine_nomod were added to the file after
it was first written, from the oracle: tests/test_oracle.py had found the compiled reference equal to the oracle in exactly
these values for these four cases, and the oracle code that computes them has not changed since.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import oracle_lib as O  # noqa: E402
import gnuspeech_b200 as g  # noqa: E402
from gnuspeech_b200 import workloads as W  # noqa: E402


def main():
    from gnuspeech_b200 import build as B
    B.build()
    B.build_oracle()
    assert O.have_reference_binary(), "needs oracle/_ref/tube_ref (built from /root/reference)"
    cases = {
        "static_a_44k": (dict(outputRate=44100.0), W.static_vowel(26, 0)),
        "static_aa_44k": (dict(outputRate=44100.0), W.static_vowel(26, 1)),
        "static_aa_22k": (dict(outputRate=22050.0), W.static_vowel(26, 1)),
        "walk_44k": (dict(outputRate=44100.0), W.random_walk(1, 51, seed=11)),
        "walk_nofric_44k": (dict(outputRate=44100.0), None),
        "walk_short_tube_down": (dict(outputRate=22050.0, length=10.0), W.random_walk(1, 31, seed=12)),
        "walk_sine_nomod": (dict(outputRate=44100.0, waveform=1, usesModulation=0), W.random_walk(1, 31, seed=13)),
        "walk_stereo": (dict(outputRate=22050.0, channels=2, balance=0.25, volume=57.0), W.random_walk(1, 31, seed=14)),
    }
    nf = W.random_walk(1, 51, seed=15)
    nf[:, 3] = 0.0          # no frication: tube.c's x10 frication gain (Appendix D.1) drops out exactly
    cases["walk_nofric_44k"] = (cases["walk_nofric_44k"][0], nf)
    out = {}
    for name, (kw, frames) in cases.items():
        ip = g.TRMInputParameters(**kw)
        r = O.synthesize(ip, frames)
        ref = O.run_reference(ip, frames)
        peak = np.abs(ref["tube"]).max()
        agree = float(np.abs(r.tube - ref["tube"]).max() / peak)
        tol = 1e-12 if frames[:, 3].max() == 0.0 else 1e-10
        assert agree <= tol, (name, agree)
        assert ref["out"].shape[0] == r.numberSamples, name
        src_agree = float(np.abs(r.samples.astype(np.float32) - ref["out"]).max() / np.abs(r.samples).max())
        assert src_agree <= 2e-7, (name, src_agree)
        out[name + "/ip"] = np.frombuffer(bytes(O.as_oracle_ip(ip)), dtype=np.uint8).copy()
        out[name + "/frames"] = frames
        out[name + "/tube"] = r.tube
        out[name + "/samples"] = r.samples
        out[name + "/max"] = np.array([r.maximumSampleValue])
        out[name + "/pcm"] = O.pcm16(ip, r.samples, r.maximumSampleValue)
        out[name + "/ref_agreement"] = np.array([agree, src_agree])
        derived = [ref["controlPeriod"], ref["sampleRate"], ref["numberTaps"], ref["padSize"]]
        assert derived == [r.info.controlPeriod, r.info.sampleRate, r.info.numberTaps, r.info.padSize], name
        out[name + "/ref_fir"] = ref["fir"]
        out[name + "/ref_derived"] = np.array(derived, np.int32)
        print("%-22s frames %3d tube %6d out %6d  oracle-vs-compiled-reference: tube %.2e  src(float) %.2e" % (
            name, frames.shape[0], r.tube.size, r.numberSamples, agree, src_agree))
    np.savez_compressed(os.path.join(HERE, "trm_golden.npz"), **out)
    print("wrote", os.path.join(HERE, "trm_golden.npz"), os.path.getsize(os.path.join(HERE, "trm_golden.npz")), "bytes")


if __name__ == "__main__":
    main()
