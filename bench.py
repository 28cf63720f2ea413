#!/usr/bin/env python
"""bench.py -- TRM synthesis throughput on B200 (BASELINE.json metric: synthesized audio-seconds per
wall-second, batched).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config 0..4] [--precision fp64|fp32] [--impl reference]

Headline workload (config.workload): BASELINE.json configs[1] per GPU -- 4096 synthetic random-walk utterances x 10 s
(2501 control frames each, male voice, 44.1 kHz mono), weak scaling: every rank synthesizes its own 4096.  `--config 4`
makes configs[4] the headline instead: ONE fixed set of 10^6 x 2 s utterances sharded over the ranks (strong scaling).

One "step" = one pass of the hot path (waveguide -> resampler -> PCM) over the whole batch.
  value     : frames resident in HBM, the three kernels launched back to back on torch's current stream, timed with
              CUDA events on that stream (max over ranks).
  e2e       : the same batch through the public C API (TRMBatchSynthesizeAsync / TRMBatchWait, include/trm.h) with
              pinned HOST buffers: every step's H2D of the frames and D2H of the PCM inside the timed region.
              e2e.ceiling = the same bytes copied with no kernels at all (TRMCopyProbe), all ranks at once.
  parity    : first / middle / last utterance of the TIMED batch against the CPU oracle (1e-9 of peak on the output
              samples in FP64, >= 80 dB in FP32, +-1 LSB on the PCM that crossed PCIe); the run FAILS otherwise.
  roofline  : dominant kernel (waveguide) -- FP-pipe bound, so the fraction is achieved FLOP/s over an FMA peak MEASURED
              live on this device (MEASURED_PEAKS.json has no CUDA-core number); roofline_src / roofline_pcm against the
              measured HBM peak, on SURVEY.md 8(d)'s minimum bytes.
  fast_mode : the same measurements in the FP32 fast mode.
  configs   : all five BASELINE configs x both precision modes (N = 1 only): value, blocking e2e, per-kernel times and
              roofline fractions.
  cpu_baseline : the CPU oracle (a C restatement of the reference, kind "port"), one utterance per thread on all host
              cores, on a bounded sample of the same workload.
--impl reference runs only that CPU arm, sized to finish in minutes, and prints its own JSON line.
--dump-outputs DIR writes what the headline's resident path computed in its last timed step (see dump_outputs) as .npy
files, so that two builds can be compared output for output on identical inputs.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# the host pipeline keeps many streams in flight; must be set before CUDA is initialised (by torch, below)
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

import numpy as np  # noqa: E402

METRIC = "synthesized audio-sec per wall-sec"
UNIT = "audio-s/s"
FLOP_PER_TUBE_SAMPLE = 390.0     # SURVEY.md 8(d): algorithmic flops per tube-rate sample
FLOP_PER_OUT_SAMPLE = 110.0      # up-sampling converter, per output sample
# DRAM traffic per unit, STATIC: dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full` capture per kernel
# (profiles/prof_r2_{fp64,fp32}_summary.txt, 4096 x 0.5 s launch), divided by that launch's units -- linear in the number of samples:
#   waveguide: bytes per tube-rate sample, resampler / PCM: bytes per output sample.  Not measured in the run it is printed in.
TRAFFIC_PER_UNIT = {"fp64": {"tube": 8.51, "src": 11.28, "pcm": 9.92}, "fp32": {"tube": 4.48, "src": 5.42, "pcm": 5.73}}
TRAFFIC_SOURCE = "static: ncu --set full DRAM bytes of a 4096 x 0.5 s launch (profiles/prof_r2_*_summary.txt), scaled by samples"


def bind_to_gpu_numa_node(torch, local_rank, world):
    """Several ranks share the host: keep this rank's threads (and with them the pinned buffers it allocates and the
    staging copies libtrm makes) on the CPUs next to its GPU, so that every GPU's PCIe traffic stays on its own socket.
    Only under torchrun; silently skipped when sysfs does not tell."""
    if world <= 1 or os.environ.get("TRM_NO_NUMA_BIND"):
        return
    try:
        pr = torch.cuda.get_device_properties(local_rank)
        path = "/sys/bus/pci/devices/%04x:%02x:%02x.0/local_cpulist" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        cpus = set()
        for part in open(path).read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            print("[bench] rank %d: bound to %d CPUs local to GPU %d" % (local_rank, len(cpus), local_rank), file=sys.stderr)
    except (OSError, ValueError, AttributeError):
        pass


def host_cores():
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            d = json.load(open(path))
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(object):
    """Samples SM clocks and throttle reasons with nvidia-smi while the timed region runs."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device, self.proc, self.lines = device, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


DUMP_BYTES = 60 * 10 ** 6          # a dump stays below 64 MB, .npy headers included


def dump_outputs(out_dir, res, maxima, seed=0):
    """Writes what a caller of the resident path receives after its last step: every utterance's maximum sample value
    (maxima.npy) and, for whole utterances drawn in a fixed seeded order while the files stay within DUMP_BYTES, their
    output-rate samples (samples.npy, in the precision mode's type) and PCM16 values (pcm.npy, as float32), back to back;
    utterances.npy and number_samples.npy say which utterances and how many samples each."""
    os.makedirs(out_dir, exist_ok=True)
    picks, lengths, samples, pcm = [], [], [], []
    size = maxima.nbytes
    for u in np.random.default_rng(seed).permutation(res.batch.n):
        smp, p, _ = res.fetch_utterance(int(u))
        cost = smp.nbytes + 4 * p.size + 16
        if size + cost > DUMP_BYTES:
            break
        size += cost
        picks.append(int(u))
        lengths.append(smp.shape[0])
        samples.append(smp)
        pcm.append(p.astype(np.float32))
    arrays = {"maxima": maxima, "utterances": np.array(picks, np.float64), "number_samples": np.array(lengths, np.float64),
              "samples": np.concatenate(samples) if samples else np.zeros(0, res.batch.sample_dtype),
              "pcm": np.concatenate(pcm) if pcm else np.zeros(0, np.float32)}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def oracle_throughput(ip, n_frames, n_utt, threads, seed, first_index):
    """Times the CPU oracle (one utterance per thread) on n_utt utterances of the workload; returns
    (audio_s_per_s, seconds)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O
    from gnuspeech_b200 import workloads as W
    frames = W.random_walk(n_utt, n_frames, seed=seed, first_index=first_index)
    t0 = time.perf_counter()
    O.synthesize_batch(ip, frames, [n_frames] * n_utt, flags=0, threads=threads)
    dt = time.perf_counter() - t0
    audio = n_utt * (n_frames - 1) / float(ip.controlRate)
    return audio / dt, dt


def run_reference_arm(args):
    """--impl reference: the reference's CPU path (oracle port of Frameworks/Tube; the Objective-C original
    cannot be built here and TRAcT/tube.c is one utterance per process), all host threads."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import gnuspeech_b200 as g
    from gnuspeech_b200 import build as B
    B.build_oracle()
    ip = g.TRMInputParameters(44100.0)
    n_frames = int(args.seconds * 250) + 1
    cores = host_cores()
    # bounded sample per step: 16 utterances per core of the same 10 s random-walk workload (~1 s wall, ~15-20 s CPU)
    n_utt = max(cores * 16, 32) if args.sample_utterances <= 0 else args.sample_utterances
    for _ in range(args.warmup):
        oracle_throughput(ip, n_frames, min(n_utt, cores), cores, args.seed, 0)
    t_total, audio_total = 0.0, 0.0
    for k in range(args.steps):
        v, dt = oracle_throughput(ip, n_frames, n_utt, cores, args.seed, k * n_utt)
        t_total += dt
        audio_total += v * dt
    value = audio_total / t_total
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * t_total / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "configs[1] sample: %d random-walk utterances x %g s per step (of 4096 x 10 s), male voice, "
                               "250 Hz control frames, 44.1 kHz mono" % (n_utt, args.seconds)},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": "%d utterances x %g s per step, one utterance per thread, reference-faithful "
                                   "per-sample wavetable rewrite" % (n_utt, args.seconds)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------------------------------
# workloads of the five BASELINE configs (per GPU)
# ------------------------------------------------------------------------------------------------------------------
def build_workload(g, W, cfg, rank, args):
    """Returns (name, ips, n_frames list, frames as a PinnedArray of float64 rows).  configs[4] is not a batch: see
    measure_sweep."""
    if cfg == 0:
        nf = 251
        pin = g.PinnedArray((nf, 16), np.float64)
        pin.array[:] = W.static_vowel(nf, 0).astype(np.float32)        # float-valued, as Monet's frame table holds them
        return "configs[0]: single utterance, static vowel /a/ 1 s, male voice, 44.1 kHz", g.TRMInputParameters(44100.0), [nf], pin
    if cfg == 1:
        n, nf = args.utterances, int(args.seconds * 250) + 1
        pin = g.PinnedArray((n * nf, 16), np.float64)
        W.random_walk(n, nf, seed=args.seed, first_index=rank * n, out=pin.array)
        name = ("configs[1]: %d random-walk utterances x %g s per GPU (%d control frames each, male voice, 250 Hz control rate, "
                "44.1 kHz mono PCM16)" % (n, args.seconds, nf))
        return name, g.TRMInputParameters(44100.0), [nf] * n, pin
    if cfg == 2:
        n, nf = 65536, 126
        pin = g.PinnedArray((n * nf, 16), np.float64)
        pin.array[:] = W.grid(range(n), nf)
        return "configs[2]: TRAcT-style static sweep, 65,536 grid points x 0.5 s (radii x velum x pitch), 44.1 kHz", g.TRMInputParameters(44100.0), [nf] * n, pin
    if cfg == 3:
        rng = np.random.default_rng(4)
        n = 256
        nfl = [int(x) for x in rng.integers(5 * 250, 60 * 250 + 1, n)]
        nfl[7], nfl[200] = 5 * 250 + 1, 60 * 250 + 1
        fr = W.random_walk_ragged(nfl, seed=9, first_index=rank * n)
        pin = g.PinnedArray(fr.shape, np.float64)
        pin.array[:] = fr
        ips = [g.TRMInputParameters(44100.0 if u % 2 == 0 else 22050.0) for u in range(n)]
        return "configs[3]: 256 random-walk utterances of 5-60 s, alternating 44.1 / 22.05 kHz", ips, nfl, pin
    raise ValueError(cfg)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default="fp64", choices=["fp64", "fp32"])
    ap.add_argument("--config", type=int, default=1, choices=[0, 1, 2, 3, 4], help="BASELINE config measured as the headline")
    ap.add_argument("--utterances", type=int, default=4096, help="configs[1]: utterances per GPU")
    ap.add_argument("--seconds", type=float, default=10.0, help="configs[1]: seconds of audio per utterance")
    ap.add_argument("--sweep-utterances", type=int, default=1000000, help="configs[4]: utterances in the whole job")
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--sample-utterances", type=int, default=0, help="CPU arm: utterances per step (0 = 16 per core)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-fast-mode", action="store_true", help="skip the FP32 fast-mode measurement of the headline")
    ap.add_argument("--no-configs", action="store_true", help="skip the all-configs section (N = 1)")
    ap.add_argument("--also-fp32", action="store_true", help=argparse.SUPPRESS)      # (round-1 flag; fast_mode is the default now)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the headline's outputs of its last timed step to DIR/*.npy "
                                                          "(rank 0; configs 0-3)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.config == 4):
        ap.error("--dump-outputs writes the outputs of the batched GPU path (configs 0-3)")

    if args.impl == "reference":
        return run_reference_arm(args)

    import torch
    import gnuspeech_b200 as g
    from gnuspeech_b200 import _native as N
    from gnuspeech_b200 import sharding
    from gnuspeech_b200 import workloads as W

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the TRM path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    bind_to_gpu_numa_node(torch, local_rank, world)
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL prints its version banner on stdout when the communicator is created; stdout carries the JSON line only
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
            warm = torch.zeros(1, device="cuda")
            dist.all_reduce(warm)
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)

    def barrier():
        if dist is not None:
            dist.barrier()

    def max_over_ranks(x):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    cores = host_cores()
    hbm_peak, hbm_src = measured_peaks()
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from gnuspeech_b200 import build as B
    B.build_oracle()                       # the checker (oracle/liboracle.so); never on the measured path
    import oracle_lib as O

    peaks = {}

    def fp_peak(precision):
        if precision not in peaks:
            L = C.CDLL(N.LIBTRM_CUDA_PATH)
            L.trm_cuda_fp_peak.argtypes = [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_double)]
            v = C.c_double(0.0)
            L.trm_cuda_fp_peak(local_rank, 0 if precision == "fp64" else 1, 3, C.byref(v))
            peaks[precision] = v.value
        return peaks[precision]

    def rooflines(precision, lay, stage_ms):
        esz = 8 if precision == "fp64" else 4
        tube_ms, src_ms, pcm_ms = stage_ms
        total = tube_ms + src_ms + pcm_ms
        peak = fp_peak(precision)
        tube_tf = FLOP_PER_TUBE_SAMPLE * float(lay.tube_samples) / (tube_ms * 1e-3) / 1e12 if tube_ms > 0 else 0.0
        tube_bytes = float(lay.total_frames) * 128 + float(lay.tube_samples) * esz
        # SURVEY.md 8(d): the converter's minimum traffic is the tube-rate signal in and the normalised PCM16 out (fused);
        # what the two kernels are written to move (R samples out, read again by the PCM pass) is reported next to it
        src_min = float(lay.tube_samples) * esz + float(lay.out_samples) * 2
        src_kernel_bytes = float(lay.tube_samples) * esz + float(lay.out_samples) * esz
        pcm_bytes = float(lay.out_samples) * (esz + 2)
        tp = TRAFFIC_PER_UNIT[precision]
        r_tube = {
            "kernel": "tube_wide_kernel<%s>" % ("double" if precision == "fp64" else "float"),
            "bound": "fp64-pipe" if precision == "fp64" else "fp32-pipe",
            "achieved": tube_tf, "peak": peak, "unit": "TFLOP/s", "frac": tube_tf / peak if peak else None,
            "peak_source": "FMA chain measured live on this device (trm_cuda_fp_peak); MEASURED_PEAKS.json has no CUDA-core peak",
            "flop_per_tube_sample": FLOP_PER_TUBE_SAMPLE, "ms_per_launch": tube_ms, "share_of_step": tube_ms / total if total else None,
            "hbm_achieved_gbs": tube_bytes / (tube_ms * 1e-3) / 1e9 if tube_ms > 0 else None,
            "algorithmic_bytes": tube_bytes, "traffic": tp["tube"] * float(lay.tube_samples), "traffic_source": TRAFFIC_SOURCE,
        }
        r_src = {
            "kernel": "src_kernel (+ pcm_kernel for the fused minimum)", "bound": "hbm",
            "achieved": src_min / ((src_ms + pcm_ms) * 1e-3) / 1e9 if src_ms + pcm_ms > 0 else None, "peak": hbm_peak, "unit": "GB/s",
            "frac": src_min / ((src_ms + pcm_ms) * 1e-3) / 1e9 / hbm_peak if src_ms + pcm_ms > 0 else None, "peak_source": hbm_src,
            "bytes_basis": "SURVEY.md 8(d) minimum: tube-rate samples read + PCM16 written, over the time of resampler + PCM kernels",
            "ms_per_launch": src_ms, "share_of_step": src_ms / total if total else None, "algorithmic_bytes": src_min,
            "kernel_bytes": src_kernel_bytes, "kernel_bytes_gbs": src_kernel_bytes / (src_ms * 1e-3) / 1e9 if src_ms > 0 else None,
            "traffic": tp["src"] * float(lay.out_samples), "traffic_source": TRAFFIC_SOURCE,
            "flops_tf": FLOP_PER_OUT_SAMPLE * float(lay.out_samples) / (src_ms * 1e-3) / 1e12 if src_ms > 0 else None,
        }
        r_pcm = {
            "kernel": "pcm_kernel", "bound": "hbm", "achieved": pcm_bytes / (pcm_ms * 1e-3) / 1e9 if pcm_ms > 0 else None, "peak": hbm_peak,
            "unit": "GB/s", "frac": pcm_bytes / (pcm_ms * 1e-3) / 1e9 / hbm_peak if pcm_ms > 0 else None, "ms_per_launch": pcm_ms,
            "share_of_step": pcm_ms / total if total else None, "algorithmic_bytes": pcm_bytes,
            "traffic": tp["pcm"] * float(lay.out_samples), "traffic_source": TRAFFIC_SOURCE,
        }
        return r_tube, r_src, r_pcm

    def check_against_oracle(precision, ips, frames, n_frames, picks, samples_of, pcm_of, max_of, what):
        """first / middle / last utterance of a timed batch against the CPU oracle; raises SystemExit on a miss"""
        off = np.concatenate(([0], np.cumsum(n_frames)))
        worst_rel, worst_lsb, worst_snr = 0.0, 0, 1e9
        for u in picks:
            ip = ips[u] if isinstance(ips, (list, tuple)) else ips
            ref = O.synthesize(ip, frames[off[u]:off[u + 1]], want_tube=False)
            y = samples_of(u)
            if y is not None and ref.numberSamples:
                y = np.asarray(y, np.float64)
                if y.shape[0] != ref.numberSamples:
                    raise SystemExit("parity FAILED (%s): utterance %d has %d samples, the oracle %d" % (what, u, y.shape[0], ref.numberSamples))
                if precision == "fp64":
                    rel = float(np.abs(y - ref.samples).max() / ref.maximumSampleValue)
                    worst_rel = max(worst_rel, rel)
                    if rel > 1e-9:
                        raise SystemExit("parity FAILED (%s): utterance %d differs from the oracle by %.3e of peak (> 1e-9)" % (what, u, rel))
                else:
                    snr = float(O.snr_db(ref.samples, y))
                    worst_snr = min(worst_snr, snr)
                    if snr < 80.0:
                        raise SystemExit("parity FAILED (%s): utterance %d SNR %.1f dB (< 80 dB)" % (what, u, snr))
            mx = max_of(u)
            tol = 1e-9 if precision == "fp64" else 2e-5
            if mx is not None and abs(mx - ref.maximumSampleValue) > tol * ref.maximumSampleValue:
                raise SystemExit("parity FAILED (%s): utterance %d maximumSampleValue %.17g vs oracle %.17g" % (what, u, mx, ref.maximumSampleValue))
            p = pcm_of(u)
            if p is not None and ref.numberSamples:
                pr = O.pcm16(ip, ref.samples, ref.maximumSampleValue).astype(np.int32)
                lsb = int(np.abs(np.asarray(p, np.int32) - pr).max())
                worst_lsb = max(worst_lsb, lsb)
                if lsb > 1:
                    raise SystemExit("parity FAILED (%s): utterance %d PCM off by %d LSB" % (what, u, lsb))
        out = {"checked_utterances": [int(u) for u in picks], "max_pcm_lsb": worst_lsb, "against": "CPU oracle (oracle/trm_oracle.c)"}
        if precision == "fp64":
            out["max_rel_err"] = worst_rel
            out["tolerance"] = "1e-9 of peak, +-1 LSB"
        else:
            out["min_snr_db"] = worst_snr
            out["tolerance"] = ">= 80 dB SNR, +-1 LSB"
        return out

    def measure_batch(precision, ips, n_frames, frames, steps, warmup, e2e_mode, with_clocks=True, dump_dir=None):
        """e2e_mode: None, "blocking" (one TRMBatchSynthesize per step) or "pipelined" (async, 3 in flight, + blocking).
        dump_dir: where dump_outputs writes the resident path's outputs of the last timed step (None: nowhere)."""
        prec = g.TRM_PRECISION_FP64 if precision == "fp64" else g.TRM_PRECISION_FP32
        n_utt = len(n_frames)
        batch = g.TRMBatch(ips, n_frames, precision=prec)
        lay = batch.layout
        audio_s = float(lay.audio_seconds)
        stream = torch.cuda.current_stream()
        sh = stream.cuda_stream
        picks = sorted(set([0, n_utt // 2, n_utt - 1]))

        # ---- value: HBM-resident inputs, kernels only --------------------------------------------------------
        res = batch.make_resident(frames, device=local_rank)
        for _ in range(warmup):
            res.run(sh)
        torch.cuda.synchronize()
        ev = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(steps)]
        sampler = ClockSampler(local_rank) if with_clocks else None
        barrier()
        torch.cuda.synchronize()
        if sampler:
            sampler.start()
        for k in range(steps):
            ev[k][0].record(stream)
            res.run_stage(N.TRM_STAGE_TUBE, sh)
            ev[k][1].record(stream)
            res.run_stage(N.TRM_STAGE_SRC, sh)
            ev[k][2].record(stream)
            res.run_stage(N.TRM_STAGE_PCM, sh)
            ev[k][3].record(stream)
        torch.cuda.synchronize()
        barrier()
        clocks = sampler.stop() if sampler else None
        total_ms = max_over_ranks(ev[0][0].elapsed_time(ev[-1][3]))
        stage_ms = [float(np.mean([ev[k][i].elapsed_time(ev[k][i + 1]) for k in range(steps)])) for i in range(3)]
        ms_per_step = total_ms / steps
        audio_all = sum_over_ranks(audio_s)
        value = audio_all / (ms_per_step * 1e-3)
        maxima = np.zeros(n_utt, np.float64)
        res.fetch(None, None, maxima, None)
        if dump_dir:
            dump_outputs(dump_dir, res, maxima)
        fetched = {u: res.fetch_utterance(u) for u in picks}          # the timed batch's own results
        res.free()
        parity = check_against_oracle(precision, ips, frames.array, n_frames, picks, lambda u: fetched[u][0],
                                      lambda u: fetched[u][1], lambda u: fetched[u][2], "resident path, %s" % precision)

        # ---- e2e: public API, host buffers, copies inside the timed region ----------------------------------
        # Every step = one TRMBatch call on this step's pinned host frames -> this step's pinned host PCM16.  A caller with a
        # stream of batches keeps three calls in flight (TRMBatchSynthesizeAsync / TRMBatchWait, include/trm.h): the PCM
        # copy-out of step k overlaps the kernels of step k+1.  All K steps' H2D, kernels and D2H complete inside the timed
        # region (the clock stops after the last TRMBatchWait).  The frames cross PCIe as float32 rows (TRM_FRAMES_F32: what
        # Monet's generator holds; the synthetic tracks are float-valued like Monet's, checked below) -- identical results,
        # half the upload.  The strictly serial form (one blocking TRMBatchSynthesize per step) is measured too.
        e2e = None
        if e2e_mode:
            f32 = g.PinnedArray(frames.array.shape, np.float32)
            f32.array[:] = frames.array
            if not np.array_equal(f32.array[:4096].astype(np.float64), frames.array[:4096]):
                raise SystemExit("the workload's frames are not float-valued")
            depth = 3 if e2e_mode == "pipelined" else 1
            batches = [batch] + [g.TRMBatch(ips, n_frames, precision=prec) for _ in range(depth - 1)]
            for b_ in batches:
                b_.set_frame_format(N.TRM_FRAMES_F32)
            pcms = [g.PinnedArray(int(lay.total_pcm_samples), np.int16) for _ in range(depth)]
            for _ in range(min(warmup, 2)):         # warms the context lanes (arenas, pinned staging)
                tk = [batches[d].synthesize_async(f32, pcm_out=pcms[d], devices=[local_rank]) for d in range(depth)]
                for t in tk:
                    t.wait()
            torch.cuda.synchronize()
            barrier()
            t0 = time.perf_counter()
            for _ in range(steps):
                batches[0].synthesize(f32, pcm_out=pcms[0], devices=[local_rank])
            torch.cuda.synchronize()
            dt_block = time.perf_counter() - t0
            barrier()
            dt_block = max_over_ranks(dt_block)
            if not np.array_equal(batches[0].maximumSampleValues, maxima):
                raise SystemExit("parity FAILED: the end-to-end and the resident path disagree")
            h2d = int(lay.total_frames) * 64
            d2h = int(lay.out_samples) * 2
            e2e = {"unit": UNIT, "h2d_bytes_per_step": h2d * world, "d2h_bytes_per_step": d2h * world,
                   "frame_format": "float32 rows (TRM_FRAMES_F32), widened by the waveguide kernel when read; bit-identical to double rows",
                   "gpu_launches_per_step": int(batches[0].kernelLaunches),
                   "blocking": {"value": audio_all / (dt_block / steps), "ms_per_step": 1e3 * dt_block / steps,
                                "api": "TRMBatchSynthesize, one blocking call per step"}}
            if e2e_mode == "pipelined":
                t0 = time.perf_counter()
                tickets, done_at = [], []
                for k in range(steps):
                    if len(tickets) == depth:
                        tickets.pop(0).wait()
                        done_at.append(time.perf_counter())
                    tickets.append(batches[k % depth].synthesize_async(f32, pcm_out=pcms[k % depth], devices=[local_rank]))
                while tickets:
                    tickets.pop(0).wait()
                    done_at.append(time.perf_counter())
                torch.cuda.synchronize()
                dt = time.perf_counter() - t0
                barrier()
                dt = max_over_ranks(dt)
                e2e.update({"value": audio_all / (dt / steps), "ms_per_step": 1e3 * dt / steps,
                            "api": "TRMBatchSynthesizeAsync / TRMBatchWait (include/trm.h), %d calls in flight, pinned host frames in, "
                                   "pinned host PCM16 out; every step's copies and kernels finish inside the timed region" % depth})
                # What the whole-run figure is made of: the first step's output is complete only after its upload, its
                # kernels and its copy-out (the latency of one step), every later one follows at the pipeline's period.
                if len(done_at) >= 3:
                    gaps = sorted(1e3 * (b_ - a_) for a_, b_ in zip(done_at[:-1], done_at[1:]))
                    period = max_over_ranks(gaps[len(gaps) // 2])
                    e2e["pipeline"] = {"first_output_ms": max_over_ranks(1e3 * (done_at[0] - t0)), "period_ms": period,
                                       "value_at_period": audio_all / (period * 1e-3),
                                       "what": "host clock at the return of each TRMBatchWait: time to the first step's complete output, "
                                               "median interval between the completions of successive steps, and the rate that interval "
                                               "corresponds to; e2e.value above is the whole run (fill and drain included) over its steps"}
                for d in range(depth):
                    if not np.array_equal(batches[d].maximumSampleValues, maxima):
                        raise SystemExit("parity FAILED: pipelined call %d and the resident path disagree" % d)
                # the copy-only ceiling of these byte counts, every rank at once
                ms = C.c_double(0.0)
                barrier()
                N.lib().TRMCopyProbe(local_rank, f32.ptr, h2d, pcms[0].ptr, d2h, max(2, steps), C.byref(ms))
                ceil_ms = max_over_ranks(ms.value)
                e2e["ceiling"] = {"value": audio_all / (ceil_ms * 1e-3), "ms_per_step": ceil_ms,
                                  "what": "TRMCopyProbe: the step's H2D and D2H bytes copied concurrently with no kernels, all ranks at once"}
                e2e["frac_of_ceiling"] = e2e["value"] / e2e["ceiling"]["value"]
            else:
                e2e.update({"value": e2e["blocking"]["value"], "ms_per_step": e2e["blocking"]["ms_per_step"], "api": e2e["blocking"]["api"]})
            # the PCM that crossed PCIe in the timed calls, against the oracle
            po, ns = batches[0].pcmOffsets, batches[0].numberSamples
            chan = [2 if (ips[u] if isinstance(ips, (list, tuple)) else ips).channels == 2 else 1 for u in range(n_utt)]
            parity["e2e"] = check_against_oracle(precision, ips, frames.array, n_frames, picks, lambda u: None,
                                                 lambda u: pcms[-1].array[po[u]:po[u] + ns[u] * chan[u]],
                                                 lambda u: float(batches[-1].maximumSampleValues[u]), "end-to-end path, %s" % precision)
            for pc in pcms:
                pc.free()
            f32.free()
        return dict(value=value, ms_per_step=ms_per_step, stage_ms=stage_ms, clocks=clocks, e2e=e2e, lay=lay,
                    audio_all=audio_all, parity=parity, launches=3 * steps)

    def measure_sweep(precision, n_total, steps=1):
        """configs[4]: ONE fixed set of n_total x 2 s utterances (walk2 tracks generated on the device, audio reduced to
        checksums on the device), sharded over the ranks by contiguous index ranges: strong scaling.  One step = one sweep
        over the whole set; `ms_total` is the time of one sweep, averaged over the `steps` timed sweeps."""
        prec = g.TRM_PRECISION_FP64 if precision == "fp64" else g.TRM_PRECISION_FP32
        ip = g.TRMInputParameters(44100.0)
        nf = 501
        lo, hi = sharding.shard_range(n_total, rank, world)
        n_local = hi - lo
        rng = np.random.default_rng(17 + rank)
        probes = sorted(set(int(x) for x in rng.integers(0, max(n_local, 1), 8))) if n_local else []
        g.sweep_synthesize(ip, nf, min(n_local, 4144), seed=args.seed, first_index=lo, precision=prec, device=local_rank)   # warm-up
        sampler = ClockSampler(local_rank)
        barrier()
        torch.cuda.synchronize()
        sampler.start()
        t0 = time.perf_counter()
        kern = 0.0
        for _ in range(steps):
            r = g.sweep_synthesize(ip, nf, n_local, seed=args.seed, first_index=lo, precision=prec, device=local_rank, probes=probes)
            kern += r["kernel_ms"] * 1e-3
        torch.cuda.synchronize()
        wall = (time.perf_counter() - t0) / steps
        barrier()
        clocks = sampler.stop()
        wall = max_over_ranks(wall)
        kern = max_over_ranks(kern / steps)
        audio = float(n_total) * (nf - 1) / 250.0
        with np.errstate(over="ignore"):
            cs = int(r["checksums"].sum(dtype=np.uint64))
        if dist is not None:
            t = torch.tensor([cs & 0xFFFFFFFF, cs >> 32], dtype=torch.int64, device="cuda")
            parts = [torch.zeros_like(t) for _ in range(world)]
            dist.all_gather(parts, t)
            cs = sum(int(p[0].item()) | (int(p[1].item()) << 32) for p in parts) & 0xFFFFFFFFFFFFFFFF
        # parity: the probed utterances against the oracle on the host twin of the device generator
        worst = 0
        for k, u in enumerate(r["probes"]):
            fr = W.walk2(1, nf, seed=args.seed, first_index=lo + int(u))
            ref = O.synthesize(ip, fr, want_tube=False)
            pr = O.pcm16(ip, ref.samples, ref.maximumSampleValue).astype(np.int32)
            lsb = int(np.abs(r["probe_pcm"][k][:ref.numberSamples].astype(np.int32) - pr).max())
            worst = max(worst, lsb)
            tol = 1e-9 if precision == "fp64" else 2e-5
            if lsb > 1 or abs(r["maxima"][int(u)] - ref.maximumSampleValue) > tol * ref.maximumSampleValue:
                raise SystemExit("parity FAILED (sweep, %s): utterance %d: PCM off by %d LSB" % (precision, lo + int(u), lsb))
        esz = 8 if precision == "fp64" else 4
        n_tube = float(n_total) * float(g.derive(ip, nf).tubeSamples)
        return {"value": audio / kern, "ms_total": kern * 1e3, "e2e": {"value": audio / wall, "unit": UNIT, "ms_total": wall * 1e3,
                "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 16 * n_total,
                "api": "TRMSweepSynthesize (include/trm.h): tracks generated on the device from (seed, index), per-utterance PCM checksum "
                       "and maximum back; wall clock around the call, all chunks"},
                "utterances": n_total, "utterances_this_rank": n_local, "audio_seconds": audio, "launches": r["launches"] * steps,
                "checksum_of_checksums": "0x%016x" % cs, "clocks": clocks,
                "parity": {"checked_utterances": [lo + int(u) for u in r["probes"]], "max_pcm_lsb": worst,
                           "against": "CPU oracle on TRMWorkloadWalk2 (the host twin of the device generator)", "tolerance": "+-1 LSB, maxima"},
                "waveguide_flops_tf": FLOP_PER_TUBE_SAMPLE * n_tube / kern / 1e12,
                "waveguide_frac_if_all_time_were_waveguide": FLOP_PER_TUBE_SAMPLE * n_tube / kern / 1e12 / fp_peak(precision),
                "hbm_bytes_generated_frames": float(n_total) * nf * 128, "esz": esz}

    # ---- headline ------------------------------------------------------------------------------------------------------
    headline_cfg = args.config
    fast = None
    if headline_cfg == 4:
        r4 = measure_sweep(args.precision, args.sweep_utterances, args.steps)
        f4 = None if args.no_fast_mode or args.precision == "fp32" else measure_sweep("fp32", args.sweep_utterances, args.steps)
        if rank == 0:
            line = {
                "metric": METRIC, "value": r4["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": 1,
                "ms_per_step": r4["ms_total"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "f64" if args.precision == "fp64" else "f32", "data": "synthetic",
                "config": {"workload": "configs[4]: %d synthetic 2 s utterances (walk2 random-walk tracks generated on the device, male voice, "
                                       "44.1 kHz mono PCM16 reduced to per-utterance checksums on the device), sharded over %d GPU(s) by "
                                       "contiguous index ranges, no collectives" % (args.sweep_utterances, world),
                           "precision_mode": args.precision, "l2": "inputs_exceed_l2 (every chunk of 4144 utterances moves 0.27 GB of frames and "
                                                                   "3.3 GB of samples through HBM)",
                           "parallelism": "utterance index range sharded across GPUs, no collectives"},
                "clocks": r4["clocks"], "e2e": r4["e2e"], "gpu_launches": r4["launches"], "parity": r4["parity"],
                "checksum_of_checksums": r4["checksum_of_checksums"], "sweep": {k: v for k, v in r4.items() if k not in ("e2e", "clocks", "parity")},
                "roofline": {"kernel": "tube_wide_kernel (the step also holds generator, resampler, PCM and checksum kernels)", "bound": "fp64-pipe" if args.precision == "fp64" else "fp32-pipe",
                             "achieved": r4["waveguide_flops_tf"], "peak": fp_peak(args.precision), "unit": "TFLOP/s",
                             "frac": r4["waveguide_frac_if_all_time_were_waveguide"], "traffic": None,
                             "note": "lower bound of the waveguide kernel's fraction: its flops over the time of ALL kernels of the sweep"},
                "cpu_baseline": None,
            }
            if f4 is not None:
                line["fast_mode"] = {"dtype": "f32", "value": f4["value"], "ms_per_step": f4["ms_total"], "e2e": f4["e2e"],
                                     "checksum_of_checksums": f4["checksum_of_checksums"], "parity": f4["parity"]}
            print(json.dumps(line))
        if dist is not None:
            dist.destroy_process_group()
        return 0

    name, ips, n_frames, frames = build_workload(g, W, headline_cfg, rank, args)
    e2e_mode = None if args.no_e2e else "pipelined"
    r = measure_batch(args.precision, ips, n_frames, frames, args.steps, args.warmup, e2e_mode,
                      dump_dir=args.dump_outputs if rank == 0 else None)
    lay = r["lay"]
    roofline, roofline_src, roofline_pcm = rooflines(args.precision, lay, r["stage_ms"])
    if not args.no_fast_mode and args.precision == "fp64":
        f = measure_batch("fp32", ips, n_frames, frames, args.steps, args.warmup, e2e_mode)
        ft, fs, fp_ = rooflines("fp32", f["lay"], f["stage_ms"])
        fast = {"dtype": "f32 (mixed: f64 pitch/phase, integer noise)", "value": f["value"], "ms_per_step": f["ms_per_step"],
                "stage_ms": {"tube": f["stage_ms"][0], "src": f["stage_ms"][1], "pcm": f["stage_ms"][2]}, "e2e": f["e2e"],
                "parity": f["parity"], "clocks": f["clocks"],
                "roofline": {"frac": ft["frac"], "achieved": ft["achieved"], "peak": ft["peak"], "unit": "TFLOP/s"},
                "roofline_src": {"frac": fs["frac"], "achieved": fs["achieved"]}, "roofline_pcm": {"frac": fp_["frac"], "achieved": fp_["achieved"]}}

    # ---- all five configs x both modes (N = 1) ---------------------------------------------------------------------------
    configs = None
    if not args.no_configs and world == 1 and headline_cfg == 1:
        configs = []
        for cfg in (0, 1, 2, 3):
            if cfg == 1:
                wl = (name, ips, n_frames, frames)
            else:
                wl = build_workload(g, W, cfg, rank, args)
            for precision in ("fp64", "fp32"):
                if cfg == 1:
                    m = r if precision == args.precision else None
                    if m is None and fast is not None:
                        m = dict(value=fast["value"], ms_per_step=fast["ms_per_step"], stage_ms=[fast["stage_ms"][k] for k in ("tube", "src", "pcm")],
                                 e2e=fast["e2e"], lay=lay, parity=fast["parity"], clocks=fast["clocks"])
                    if m is None:
                        continue
                else:
                    m = measure_batch(precision, wl[1], wl[2], wl[3], 2, 1, None if args.no_e2e else "blocking")
                rt, rs, rp = rooflines(precision, m["lay"], m["stage_ms"])
                configs.append({
                    "config": cfg, "workload": wl[0], "precision_mode": precision, "value": m["value"], "unit": UNIT,
                    "ms_per_step": m["ms_per_step"], "audio_seconds": float(m["lay"].audio_seconds),
                    "stage_ms": {"tube": m["stage_ms"][0], "src": m["stage_ms"][1], "pcm": m["stage_ms"][2]},
                    "e2e": None if m["e2e"] is None else {"value": m["e2e"]["value"], "ms_per_step": m["e2e"]["ms_per_step"], "api": m["e2e"]["api"],
                                                          "h2d_bytes_per_step": m["e2e"]["h2d_bytes_per_step"], "d2h_bytes_per_step": m["e2e"]["d2h_bytes_per_step"]},
                    "roofline_frac": {"waveguide": rt["frac"], "src_plus_pcm_on_minimum_bytes": rs["frac"], "pcm": rp["frac"]},
                    "parity": m["parity"], "clocks": m["clocks"]})
            if cfg != 1:
                wl[3].free()
        for precision in ("fp64", "fp32"):
            s4 = measure_sweep(precision, args.sweep_utterances)
            configs.append({"config": 4, "workload": "configs[4]: %d x 2 s, tracks generated on the device, checksum sink" % args.sweep_utterances,
                            "precision_mode": precision, "value": s4["value"], "unit": UNIT, "ms_per_step": s4["ms_total"],
                            "audio_seconds": s4["audio_seconds"], "e2e": {"value": s4["e2e"]["value"], "ms_per_step": s4["e2e"]["ms_total"], "api": s4["e2e"]["api"],
                                                                          "h2d_bytes_per_step": 0, "d2h_bytes_per_step": s4["e2e"]["d2h_bytes_per_step"]},
                            "roofline_frac": {"waveguide_lower_bound": s4["waveguide_frac_if_all_time_were_waveguide"]},
                            "checksum_of_checksums": s4["checksum_of_checksums"], "parity": s4["parity"], "clocks": s4["clocks"]})

    # ---- CPU baseline on a bounded sample (rank 0, N=1 only) ------------------------------------------------
    cpu = None
    if not args.no_cpu_baseline and rank == 0 and world == 1:
        ip1 = g.TRMInputParameters(44100.0)
        nf1 = int(args.seconds * 250) + 1
        n_s = min(args.utterances, max(16 * cores, 32))           # ~15-20 s of CPU work
        v, dt = oracle_throughput(ip1, nf1, n_s, cores, args.seed, 0)
        cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "seconds": dt,
               "sample": "%d of the %d utterances x %g s of configs[1], one utterance per thread, reference-faithful per-sample "
                         "wavetable rewrite" % (n_s, args.utterances, args.seconds)}

    if rank == 0:
        esz = 8 if args.precision == "fp64" else 4
        tube_ms, src_ms, pcm_ms = r["stage_ms"]
        line = {
            "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64" if args.precision == "fp64" else "f32",
            "data": "synthetic",
            "config": {"workload": name,
                       "utterances_per_gpu": len(n_frames), "audio_seconds_per_gpu": float(lay.audio_seconds),
                       "tube_samples_per_gpu": int(lay.tube_samples), "out_samples_per_gpu": int(lay.out_samples),
                       "precision_mode": args.precision + (" conformance (<= 1e-9 of the reference; checked in this run, see parity)" if args.precision == "fp64" else " fast"),
                       "l2": "inputs_exceed_l2 (frames %.2f GB + tube-rate %.2f GB per step >> 126 MB)" % (
                           lay.total_frames * 128 / 1e9, lay.tube_samples * esz / 1e9),
                       "parallelism": "utterances sharded across GPUs, no collectives"},
            "clocks": r["clocks"],
            "e2e": r["e2e"],
            "gpu_launches": r["launches"],
            "stage_ms": {"tube": tube_ms, "src": src_ms, "pcm": pcm_ms},
            "parity": r["parity"],
            "roofline": roofline, "roofline_src": roofline_src, "roofline_pcm": roofline_pcm,
            "cpu_baseline": cpu,
        }
        if fast is not None:
            line["fast_mode"] = fast
        if configs is not None:
            line["configs"] = configs
        print(json.dumps(line))
    frames.free()
    if dist is not None:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
