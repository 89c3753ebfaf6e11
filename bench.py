#!/usr/bin/env python
"""bench.py — the reference's headline metric on its named configurations, one JSON line on rank 0.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload mel|cluster] [--impl ours|reference] [--dump-outputs DIR]

Main line (BASELINE.json configs[1], the configuration the metric is quoted on):
    log-mel of 1 h of synthetic 16 kHz mono audio, 25 ms / 10 ms frames, 512-point FFT, 80 mels -> [360 001 x 80].
    A step = one pass over the hour.  `value` = audio-hours/s with audio and output resident in HBM (CUDA events on the
    launching stream, exactly K steps); `sustained` = the same launch repeated for >= 1 s; `e2e` = the same through
    fa_mel_compute with pinned HOST buffers (H2D and D2H inside); `e2e_i16` = int16 PCM through fa_audio_to_mel (the
    AudioConverter stage on the device: half the H2D bytes); `copy_floor` = the bare copies of the same bytes.
    The transform runs in float32 like the reference's vDSP_DFT (FA_MEL_PRECISION_F32: packed FFMA2, two frames per
    warp); the run itself checks that choice against the FP64-transform path over the WHOLE hour (`parity`, bar 1e-4,
    a failed bar makes the run report the FP64 path as `value`) and reports the FP64 path's numbers under `f64_transform`.
Attached sub-objects, each with its own parity field:
    `cluster` configs[2]: 10 000 x 256 embeddings -> normalise + AHC + cut + VBx + centroids + assignment (per GPU, weak).
    `c4`      configs[3]: 512 clips x 30 s SHARDED over the ranks (contiguous blocks), strong scaling, host buffers.
    `c5`      configs[4]: 64 meetings x 5 000 x 256 SHARDED over the ranks (LPT), labels gathered over NCCL and hashed
              against goldens produced by the compiled reference (tests/golden/c5_meetings.json): `labels_equal_ref`.
    `streaming`: p50 / p99 latency of small `.prePadded` calls (the production callers' shape).
--dump-outputs DIR: after the timed steps rank 0 writes what the last timed step computed, as DIR/<name>.npy: the log-mel
rows of the headline path (a fixed sample of MEL_DUMP_ROWS frames, drawn with seed 0, float32) and the cluster labels
(float64) and centroids (float64) of the 10 000 x 256 problem.  Inputs are seeded, so two builds compare output for output.
With N > 1 (torchrun) units are independent: no data-path collective; NCCL carries the barrier, the MAX-reduction of
times and the gather of labels / checksums.  Timing: barrier + device sync on both sides, MAX over ranks.

--impl reference: the reference's CPU implementation of the path on the host cores, rank 0 only — for `mel` the
float32-FFT port of AudioMelSpectrogram vectorised across frames (oracle/oracle_mel_fast.cpp; no Swift toolchain
exists), for `cluster` the UNMODIFIED FastClusterWrapper.cpp (oracle/_ref) plus the oracle port of the Swift stages.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import sys
import threading
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the tree may be read-only: nothing is written next to the sources

MEL_SAMPLES = 57_600_000
MEL_FRAMES = 360_001
N_MELS = 80
MEL_BYTES_PER_HOUR = 4 * MEL_SAMPLES + 4 * MEL_FRAMES * N_MELS            # 345 600 320 B (SURVEY §8d)
CLUSTER_N, CLUSTER_D, CLUSTER_R, CLUSTER_K = 10_000, 256, 128, 8
AHC_BYTES = 8.0 * CLUSTER_D * CLUSTER_N * CLUSTER_N                       # 2.048e11 B (SURVEY §8d)
C4_CLIPS, C4_SAMPLES = 512, 480_000
C5_MEETINGS, C5_N = 64, 5_000
MEL_TOL = 1e-4
MEL_DUMP_ROWS = 65_536                                                    # 21 MB of the 115 MB output


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """SM clock, power and throttle reasons sampled IN PROCESS through NVML every ~2 ms while `active` (a 10 ms timed
    region is invisible to a 100 ms nvidia-smi poll)."""

    def __init__(self, index: int):
        self.rows, self.active, self.stop_flag, self.h, self.nv = [], False, False, None, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_sm = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.t = threading.Thread(target=self._run, daemon=True)
            self.t.start()
        except Exception:
            self.h = None

    def _run(self):
        nv = self.nv
        while not self.stop_flag:
            if self.active:
                try:
                    self.rows.append((nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM),
                                      nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0,
                                      nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)))
                except Exception:
                    pass
            time.sleep(0.002)

    def __enter__(self):
        self.active = True
        return self

    def __exit__(self, *a):
        self.active = False

    def summary(self):
        self.stop_flag = True
        if self.h is None or not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        nv = self.nv
        names = {"hw_slowdown": nv.nvmlClocksEventReasonHwSlowdown, "hw_thermal_slowdown": nv.nvmlClocksEventReasonHwThermalSlowdown,
                 "sw_thermal_slowdown": nv.nvmlClocksEventReasonSwThermalSlowdown, "sw_power_cap": nv.nvmlClocksEventReasonSwPowerCap}
        bits = 0
        for r in self.rows:
            bits |= int(r[2])
        sm = [r[0] for r in self.rows]
        return {"sm_mhz": float(np.median(sm)), "sm_min_mhz": float(min(sm)), "sm_max_mhz": self.max_sm,
                "power_w_max": float(max(r[1] for r in self.rows)), "reasons": sorted(k for k, v in names.items() if bits & v),
                "samples": len(sm), "how": "NVML in process, 2 ms period, timed regions only"}


# ------------------------------------------------------------------------------------------------ CPU arms
def host_threads() -> int:
    return max(1, min(os.cpu_count() or 1, 64))


def cpu_mel(audio: np.ndarray, threads: int, repeats: int = 1, fast: bool = True):
    """AudioMelSpectrogram on `threads` host threads: the audio cut into 30 s clips, every clip processed `repeats`
    times, one instance and one output buffer per thread (ctypes releases the GIL inside the C++ call).
    fast=True: the float32-FFT port vectorised across frames (oracle_mel_fast.cpp — the reference's arithmetic);
    fast=False: the parity oracle itself (float64 DFT rounded once, scalar)."""
    import ctypes as C
    from oracle import oracle as O
    L = O.lib()
    L.oracle_tune_allocator()
    cfg = O.mel_config(n_mels=N_MELS)
    clip = 480_000
    pieces = [np.ascontiguousarray(audio[i:i + clip]) for i in range(0, audio.size, clip)] * repeats
    shares = [s for s in (pieces[t::threads] for t in range(threads)) if s]
    O.mel_fast_flat_transposed(cfg, pieces[0][:16000])           # sets argtypes, warms the thread-local instance
    cap = (1 + (clip + 112) // 160) * N_MELS

    def work(share):
        out = np.empty(cap, np.float32)
        ml, nf = C.c_int64(), C.c_int64()
        for p in share:
            if fast:
                L.oracle_mel_fast_flat_transposed(C.byref(cfg), p.ctypes.data, p.size, 0.0, out.ctypes.data, cap, C.byref(ml))
            else:
                L.oracle_mel_compute_flat_transposed(C.byref(cfg), p.ctypes.data, p.size, 0.0, 0, -1, out.ctypes.data, cap,
                                                     C.byref(ml), C.byref(nf))
        return 0

    t0 = time.perf_counter()
    with ThreadPoolExecutor(len(shares)) as ex:
        list(ex.map(work, shares))
    dt = time.perf_counter() - t0
    return (repeats * audio.size / 16000.0 / 3600.0) / dt, dt


def cpu_mel_arm(audio: np.ndarray, threads: int, budget_s: float = 8.0):
    """Bounded sample of the mel workload on all host threads: repeats sized so that the arm runs ~budget_s."""
    v, dt = cpu_mel(audio, threads, 1)
    repeats = int(max(1, min(64, budget_s / max(dt, 1e-3))))
    v, dt = cpu_mel(audio, threads, repeats)
    return v, dt, repeats


def cpu_cluster(emb, rho, psi):
    from oracle import oracle as O
    t0 = time.perf_counter()
    res = O.diarize_cluster(emb, rho, psi, use_ref=O.ref_available())
    dt = time.perf_counter() - t0
    return emb.shape[0] / dt, dt, ("reference" if O.ref_available() else "port"), res


# ------------------------------------------------------------------------------------------------ GPU arms
def _timed_steps(mel, fn, steps, dist, sharding):
    sharding.barrier(dist)
    mel.timer_start()
    for _ in range(steps):
        fn()
    ms = mel.timer_stop_ms()
    sharding.barrier(dist)
    return sharding.all_reduce_max(dist, ms)


def _timed_wall(fn, steps, dist, sharding, _lib):
    sharding.barrier(dist)
    t0 = time.perf_counter()
    for _ in range(steps):
        fn()
    _lib.synchronize()
    dt = time.perf_counter() - t0
    sharding.barrier(dist)
    return sharding.all_reduce_max(dist, dt)


def bench_mel(args, dist, clocks):
    import ctypes as C
    from fluidaudio_b200 import _lib, sharding, synth
    from fluidaudio_b200.mel import AudioMelSpectrogram, Precision
    audio = synth.tone_noise_audio(MEL_SAMPLES, seed=7)      # BASELINE's signal on every rank (weak scaling: one hour per GPU)
    mel = AudioMelSpectrogram(n_mels=N_MELS, precision=Precision.f32)
    mel64 = AudioMelSpectrogram(n_mels=N_MELS, precision=Precision.f64)
    pin_in = _lib.PinnedArray(MEL_SAMPLES, np.float32)
    pin_in.array[:] = audio
    pin_i16 = _lib.PinnedArray(MEL_SAMPLES, np.int16)
    pin_i16.array[:] = np.round(audio * 32767.0).astype(np.int16)
    pin_out = _lib.PinnedArray(MEL_FRAMES * N_MELS, np.float32)
    d_in = _lib.DeviceBuffer(MEL_SAMPLES * 4 + 64)
    d_out = _lib.DeviceBuffer(MEL_FRAMES * N_MELS * 4)
    d_in.upload(audio)
    K, W = args.steps, args.warmup
    # ---- kernel-only: inputs resident in HBM (345.6 MB touched per step > 126 MB L2: nothing survives a step) ----
    step = lambda: mel.compute_device(d_in, MEL_SAMPLES, d_out)
    step64 = lambda: mel64.compute_device(d_in, MEL_SAMPLES, d_out)
    for _ in range(W):
        step()
    _lib.synchronize()
    launches0 = _lib.kernel_launch_count()
    with clocks:
        dev_ms = _timed_steps(mel, step, K, dist, sharding)
    launches = _lib.kernel_launch_count() - launches0
    got32 = d_out.download((MEL_FRAMES, N_MELS), np.float32)
    # sustained: the same launch back to back for >= ~1.2 s
    reps = int(max(K, min(20000, 1200.0 / max(dev_ms / K, 1e-3))))
    with clocks:
        sus_ms = _timed_steps(mel, step, reps, dist, sharding)
    # FP64-transform path (the library default), same K steps
    for _ in range(W):
        step64()
    with clocks:
        dev64_ms = _timed_steps(mel64, step64, K, dist, sharding)
    got64 = d_out.download((MEL_FRAMES, N_MELS), np.float32)
    diff = float(np.abs(got32 - got64).max())
    # ---- end to end through the C ABI with host buffers --------------------------------------------------------
    e2e = lambda: mel.compute_flat_transposed(pin_in.array, out=pin_out.array)
    for _ in range(W):
        e2e()
    with clocks:
        e2e_s = _timed_wall(e2e, K, dist, sharding, _lib)
    assert np.array_equal(pin_out.array.reshape(MEL_FRAMES, N_MELS), got32), "host-buffer path differs from the resident one"
    e2e16 = lambda: mel.compute_from_pcm(pin_i16.array, 16000.0, out=pin_out.array)
    for _ in range(W):
        e2e16()
    e2e16_s = _timed_wall(e2e16, K, dist, sharding, _lib)
    i16_diff = float(np.abs(pin_out.array.reshape(MEL_FRAMES, N_MELS)[:6000] - got32[:6000]).max())   # 16-bit quantised input
    # bare copies of the same bytes on two streams: the floor under the end-to-end numbers; each direction alone as well,
    # all ranks copying at the same time (at N = 8 four GPUs share a socket: this names the limiter of the e2e scaling)
    L = _lib.load()
    ms = C.c_float()
    floor = {}
    nb_out = 4 * MEL_FRAMES * N_MELS
    for name, src, nb_in, nb_o in (("f32", pin_in, 4 * MEL_SAMPLES, nb_out), ("i16", pin_i16, 2 * MEL_SAMPLES, nb_out),
                                    ("h2d_only", pin_in, 4 * MEL_SAMPLES, 0), ("d2h_only", pin_in, 0, nb_out)):
        sharding.barrier(dist)
        _lib.check(L.fa_memcpy_probe(src.array.ctypes.data, nb_in, pin_out.array.ctypes.data, nb_o,
                                     max(3, min(K, 10)), C.byref(ms)), "fa_memcpy_probe")
        floor[name] = sharding.all_reduce_max(dist, float(ms.value))
    numa = sharding.numa_node_of(pin_in.array.ctypes.data)
    ms_per_step = dev_ms / K
    hours = dist.world * 1.0
    peak, peak_src = measured_peaks()
    achieved = MEL_BYTES_PER_HOUR / (ms_per_step * 1e-3) / 1e9
    out = {
        "metric": "audio-hours/s", "value": hours / (ms_per_step * 1e-3), "unit": "audio-hours/s",
        "ms_per_step": ms_per_step, "dtype": "f32",
        "sustained": {"value": hours / (sus_ms / reps * 1e-3), "ms_per_step": sus_ms / reps, "steps": reps,
                      "seconds": sus_ms * 1e-3},
        "f64_transform": {"value": hours / (dev64_ms / K * 1e-3), "ms_per_step": dev64_ms / K,
                          "roofline_frac": MEL_BYTES_PER_HOUR / (dev64_ms / K * 1e-3) / 1e9 / peak,
                          "note": "FA_MEL_PRECISION_F64 (library default): DFT in FP64 rounded once, one frame per warp"},
        "parity": {"bar": MEL_TOL, "max_abs_f32_vs_f64_transform_full_hour": diff, "values_compared": int(got32.size),
                   "max_abs_i16_pcm_vs_f32_pcm_first_minute": i16_diff},
        "e2e": {"value": hours / (e2e_s / K), "unit": "audio-hours/s", "ms_per_step": e2e_s / K * 1e3,
                "h2d_bytes_per_step": 4 * MEL_SAMPLES, "d2h_bytes_per_step": 4 * MEL_FRAMES * N_MELS,
                "host_buffers": "pinned (fa_host_alloc)", "api": "fa_mel_compute",
                "copy_floor_ms": floor["f32"], "of_copy_floor": floor["f32"] / (e2e_s / K * 1e3),
                "copy_floor_h2d_only_ms": floor["h2d_only"], "copy_floor_d2h_only_ms": floor["d2h_only"],
                "copy_floor_note": "fa_memcpy_probe: bare cudaMemcpyAsync of the same bytes on two streams, all ranks at once, MAX over ranks",
                "pinned_input_numa_node": numa},
        "e2e_i16": {"value": hours / (e2e16_s / K), "unit": "audio-hours/s", "ms_per_step": e2e16_s / K * 1e3,
                    "h2d_bytes_per_step": 2 * MEL_SAMPLES, "d2h_bytes_per_step": 4 * MEL_FRAMES * N_MELS,
                    "api": "fa_audio_to_mel (int16 PCM, 16 kHz mono: widening on the device)",
                    "copy_floor_ms": floor["i16"], "of_copy_floor": floor["i16"] / (e2e16_s / K * 1e3)},
        "gpu_launches": int(launches),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": 316.8e6, "traffic_source": "ncu --set full, profiles/r02_summary.txt: dram read 230.5 MB + write "
                     "86.3 MB per launch (the tail of the output is still in L2 at kernel end)",
                     "kernel": "mel512_kernel<8, f32x2>", "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": MEL_BYTES_PER_HOUR},
        "config": {"workload": "log-mel STFT, 1 h synthetic 16 kHz mono, 25 ms/10 ms frames, nFFT 512, 80 mels, per GPU",
                   "samples": MEL_SAMPLES, "frames": MEL_FRAMES, "n_mels": N_MELS, "transform": "float32 (FA_MEL_PRECISION_F32)",
                   "l2": "inputs+outputs 345.6 MB per step exceed the 126 MB L2 (no flush needed)",
                   "parallelism": f"dp{dist.world}: one process per GPU, independent clips, no data-path collective"},
    }
    out["parity"]["ok"] = bool(diff <= MEL_TOL)
    if diff > MEL_TOL:   # the float32 headline is void: fall back to reporting the FP64-transform path as the value
        out["parity"]["note"] = "float32 transform exceeded the bar on this signal: value / roofline below are the FP64 transform's"
        out["value"], out["ms_per_step"] = out["f64_transform"]["value"], out["f64_transform"]["ms_per_step"]
        out["roofline"]["frac"] = out["f64_transform"]["roofline_frac"]
        out["roofline"]["achieved"] = out["roofline"]["frac"] * peak
        out["roofline"]["kernel"] = "mel512_kernel<8, double>"
    return out, audio, got32, (got32 if diff <= MEL_TOL else got64)


def bench_streaming(args):
    """Latency of the production callers' small `.prePadded` calls (SortformerDiarizer.swift:857-905 streams 10 080-sample
    chunks, StreamingEouAsrManager 2 560 / 20 480: EouChunkSizeFrameCountTests.swift:10-41), host buffers in and out."""
    from fluidaudio_b200 import synth
    from fluidaudio_b200.mel import AudioMelSpectrogram, PaddingMode, Precision
    out = {}
    mel = AudioMelSpectrogram(n_mels=128, precision=Precision.f32)
    for n in (2560, 10080, 20480):
        a = synth.tone_noise_audio(n, seed=n)
        buf = np.empty(mel.frame_count(n, PaddingMode.pre_padded) * 128, np.float32)
        for _ in range(20):
            mel.compute_flat_transposed(a, padding_mode=PaddingMode.pre_padded, out=buf)
        ts = []
        for _ in range(300):
            t0 = time.perf_counter()
            mel.compute_flat_transposed(a, last_audio_sample=0.1, padding_mode=PaddingMode.pre_padded, out=buf)
            ts.append(time.perf_counter() - t0)
        ts = np.sort(np.array(ts)) * 1e6
        out[str(n)] = {"frames": int(buf.size // 128), "p50_us": float(ts[len(ts) // 2]), "p99_us": float(ts[int(len(ts) * 0.99)]),
                       "min_us": float(ts[0])}
    out["api"] = "fa_mel_compute, .prePadded, 128 mels, pageable host buffers, 300 calls each (wall clock incl. ctypes)"
    return out


def bench_cluster(args, dist):
    from fluidaudio_b200 import _lib, sharding, synth
    from fluidaudio_b200.clustering import OfflineClusterer
    steps = args.steps
    emb, _ = synth.speaker_embeddings(CLUSTER_N, CLUSTER_D, CLUSTER_K, sigma=0.02, seed=42 + dist.rank)
    rho, psi = synth.synthetic_plda(emb, CLUSTER_R)
    pin_e = _lib.PinnedArray(emb.shape, np.float32); pin_e.array[:] = emb
    pin_r = _lib.PinnedArray(rho.shape, np.float64); pin_r.array[:] = rho
    c = OfflineClusterer(psi=psi)
    for _ in range(max(1, min(args.warmup, 3))):
        res = c.cluster(pin_e.array, pin_r.array)
    sharding.barrier(dist)
    launches0 = _lib.kernel_launch_count()
    t0 = time.perf_counter()
    dev_ms, ahc_ms = 0.0, 0.0
    for _ in range(steps):
        res = c.cluster(pin_e.array, pin_r.array)
        i = res.info
        dev_ms += i["ms_normalize"] + i["ms_ahc"] + i["ms_cut"] + i["ms_vbx"] + i["ms_assign"]
        ahc_ms += i["ms_ahc"]
    e2e_s = time.perf_counter() - t0
    launches = _lib.kernel_launch_count() - launches0
    sharding.barrier(dist)
    e2e_s = sharding.all_reduce_max(dist, e2e_s)
    dev_ms = sharding.all_reduce_max(dist, dev_ms)
    peak, peak_src = measured_peaks()
    achieved = AHC_BYTES / (ahc_ms / steps * 1e-3) / 1e9
    n_total = dist.world * CLUSTER_N
    out = {
        "metric": "embeddings/s", "value": n_total / (dev_ms / steps * 1e-3), "unit": "embeddings/s",
        "ms_per_step": dev_ms / steps, "dtype": "f64",
        "e2e": {"value": n_total / (e2e_s / steps), "unit": "embeddings/s", "ms_per_step": e2e_s / steps * 1e3,
                "h2d_bytes_per_step": int(emb.nbytes + rho.nbytes), "d2h_bytes_per_step": int(4 * CLUSTER_N + 32 * (CLUSTER_N - 1)),
                "host_buffers": "pinned (fa_host_alloc)", "api": "fa_diarize_cluster"},
        "gpu_launches": int(launches),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": 42.3e6, "traffic_source": "ncu --set full, profiles/r01c_summary.txt: ahc_merge_kernel dram "
                     "read 41.3 MB + write 1.0 MB per launch (+ 20.5 MB read by ahc_init_nn_kernel)",
                     "kernel": "ahc_merge_kernel (+ ahc_init_nn_kernel)", "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": AHC_BYTES,
                     "note": "node vectors are resident in shared memory, so algorithmic bytes are served on-chip; "
                             "the loop is bound by N-1 dependent steps (latency), see DESIGN.md"},
        "stages_ms": {k: res.info[k] for k in ("ms_normalize", "ms_ahc", "ms_cut", "ms_vbx", "ms_assign", "ms_total")},
        "config": {"workload": "offline diarization backend: 10 000 x 256-d embeddings (8 speakers), cosine-normalise + "
                               "centroid AHC (thr 0.6) + cut + VBx (Fa 0.07, Fb 0.8, <=20 it) + centroids + argmax, per GPU",
                   "n": CLUSTER_N, "dim": CLUSTER_D, "rho_dim": CLUSTER_R,
                   "parallelism": f"dp{dist.world}: one process per GPU, independent embedding sets"},
    }
    # parity at every N: rank r's labels hashed against the golden of seed 42 (rank 0) — other seeds are checked through
    # determinism (two runs, identical labels)
    golden = json.load(open(os.path.join(ROOT, "tests", "golden", "ahc_large.json")))["c3_10000x256_seed42"]
    ok = 1.0
    if dist.rank == 0:
        ok = 1.0 if hashlib.sha256(np.ascontiguousarray(res.labels, np.int32).tobytes()).hexdigest() == golden["final_labels_sha256"] else 0.0
    again = c.cluster(pin_e.array, pin_r.array)
    same = 1.0 if np.array_equal(again.labels, res.labels) else 0.0
    out["labels_equal_ref"] = bool(sharding.all_reduce_sum(dist, ok if dist.rank == 0 else 0.0) == 1.0)
    out["labels_deterministic_all_ranks"] = bool(sharding.all_reduce_sum(dist, same) == dist.world)
    return out, (emb, rho, psi, res)


def _stats(ts):
    ts = sorted(ts)
    return {"min": ts[0], "median": ts[len(ts) // 2], "max": ts[-1], "reps": len(ts)}


def bench_c4(args, dist):
    """BASELINE configs[3]: 512 clips x 30 s, clip i generated from seed i, sharded in contiguous blocks over the ranks,
    each rank running fa_mel_compute_batch from pinned host memory to pinned host memory.  Strong scaling: the job is the
    512 clips whatever N.  Parity at every N: per-clip SHA-256 of the output rows are gathered over the process group and
    rank 0 recomputes the first clip of every rank's shard on its own GPU (a clip's result may not depend on its batch)."""
    from fluidaudio_b200 import _lib, sharding, synth
    from fluidaudio_b200.mel import AudioMelSpectrogram, Precision
    mel = AudioMelSpectrogram(n_mels=N_MELS, precision=Precision.f32)
    mine = sharding.contiguous_shard(C4_CLIPS, dist.rank, dist.world)
    count = len(mine)
    T = mel.frame_count(C4_SAMPLES)
    pin_in = _lib.PinnedArray((count * C4_SAMPLES,), np.float32)
    for j, i in enumerate(mine):
        pin_in.array[j * C4_SAMPLES:(j + 1) * C4_SAMPLES] = synth.tone_noise_audio(C4_SAMPLES, seed=i)
    offsets = np.arange(count + 1, dtype=np.int64) * C4_SAMPLES
    pin_out = _lib.PinnedArray((count * T * N_MELS,), np.float32)
    run = lambda: mel.compute_batch(None, packed_audio=pin_in.array, offsets=offsets, out=pin_out.array)
    for _ in range(2):
        run()
    ts = [_timed_wall(run, 1, dist, sharding, _lib) for _ in range(5)]
    st = _stats(ts)
    out = pin_out.array.reshape(count, T * N_MELS)
    digests = np.stack([np.frombuffer(hashlib.sha256(out[j].tobytes()).digest(), np.uint8) for j in range(count)])
    allhash = sharding.gather_bytes(dist, digests, [len(sharding.contiguous_shard(C4_CLIPS, r, dist.world)) for r in range(dist.world)])
    checked = equal = 0
    if dist.is_root:
        for r in range(dist.world):
            i = sharding.contiguous_shard(C4_CLIPS, r, dist.world)[0]
            a = synth.tone_noise_audio(C4_SAMPLES, seed=i)
            single, _, _ = mel.compute_flat_transposed(a)
            checked += 1
            equal += int(hashlib.sha256(single.tobytes()).digest() == allhash[i].tobytes())
    hours = C4_CLIPS * 30.0 / 3600.0
    return {"workload": "configs[3]: 512 clips x 30 s sharded over the ranks (contiguous blocks), fa_mel_compute_batch, "
                        "pinned host buffers in and out", "scaling": "strong", "clips_per_rank": count,
            "e2e": {"value": hours / st["median"], "unit": "audio-hours/s", "ms": {k: v * 1e3 for k, v in st.items() if k != "reps"},
                    "reps": st["reps"], "h2d_bytes_per_rank": int(4 * count * C4_SAMPLES), "d2h_bytes_per_rank": int(4 * count * T * N_MELS)},
            "clips_hashed": int(C4_CLIPS if dist.is_root else count), "clips_recomputed_on_rank0": checked, "clips_equal": equal}


def bench_c5(args, dist):
    """BASELINE configs[4]: 64 meetings x 5 000 x 256 (seed = meeting index), partitioned over the ranks by LPT on 8 d N^2,
    each rank running fa_diarize_cluster_batch; labels gathered over the process group (NCCL) and every meeting's labels
    hashed against tests/golden/c5_meetings.json — goldens produced by the compiled reference fastcluster + the oracle
    port of the Swift stages.  Strong scaling."""
    from fluidaudio_b200 import _lib, sharding, synth
    from fluidaudio_b200.clustering import OfflineClusterer
    parts = sharding.lpt_partition([sharding.ahc_cost(C5_N, CLUSTER_D)] * C5_MEETINGS, dist.world)
    mine = parts[dist.rank]
    embs, rhos, psi = [], [], None
    for m in mine:
        e, _ = synth.speaker_embeddings(C5_N, CLUSTER_D, 4, weights=(0.4, 0.3, 0.2, 0.1), sigma=0.02, seed=m)
        r, psi = synth.synthetic_plda(e, CLUSTER_R)
        embs.append(e); rhos.append(r)
    pin_e = _lib.PinnedArray((len(mine) * C5_N, CLUSTER_D), np.float32); pin_e.array[:] = np.concatenate(embs)
    pin_r = _lib.PinnedArray((len(mine) * C5_N, CLUSTER_R), np.float64); pin_r.array[:] = np.concatenate(rhos)
    offs = np.arange(len(mine) + 1, dtype=np.int64) * C5_N
    c = OfflineClusterer(psi=psi)
    box = {}

    def run():
        box["labels"], box["infos"] = c.cluster_batch(pin_e.array, pin_r.array, offs)
    run()
    ts = [_timed_wall(run, 1, dist, sharding, _lib) for _ in range(5)]
    st = _stats(ts)
    counts = [len(p) * C5_N for p in parts]
    gathered = sharding.gather_labels(dist, box["labels"], counts)
    equal = None
    if dist.is_root:
        golden = {g["meeting"]: g["final_labels_sha256"] for g in
                  json.load(open(os.path.join(ROOT, "tests", "golden", "c5_meetings.json")))["meetings"]}
        equal, pos = 0, 0
        for r in range(dist.world):
            for m in parts[r]:
                lab = np.ascontiguousarray(gathered[pos:pos + C5_N], np.int32)
                equal += int(hashlib.sha256(lab.tobytes()).hexdigest() == golden[m])
                pos += C5_N
    ahc = [i["ms_ahc"] for i in box["infos"]]
    return {"workload": "configs[4]: 64 meetings x 5 000 x 256 sharded over the ranks (LPT), fa_diarize_cluster_batch, labels "
                        "gathered over the process group", "scaling": "strong", "meetings_per_rank": len(mine),
            "e2e": {"value": C5_MEETINGS * C5_N / st["median"], "unit": "embeddings/s",
                    "ms": {k: v * 1e3 for k, v in st.items() if k != "reps"}, "reps": st["reps"]},
            "ahc_ms_per_meeting": {"min": float(min(ahc)), "max": float(max(ahc))},
            "labels_equal_ref": equal, "meetings": C5_MEETINGS,
            "golden": "tests/golden/c5_meetings.json (compiled reference fastcluster + oracle port of the Swift stages)"}


def dump_outputs(out_dir, mel_rows, cluster_res):
    """The last timed step's results as .npy files (float32 / float64): a seeded sample of the log-mel rows, and the
    cluster labels and centroids."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"cluster_labels": np.asarray(cluster_res.labels, np.float64),
              "cluster_centroids": np.asarray(cluster_res.centroids, np.float64)}
    if mel_rows is not None:
        rows = np.sort(np.random.default_rng(0).choice(MEL_FRAMES, MEL_DUMP_ROWS, replace=False))
        arrays["mel_rows_sample"] = np.ascontiguousarray(mel_rows[rows], np.float32)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", choices=["mel", "cluster"], default="mel")
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--only-main", action="store_true", help="skip the c4 / c5 / streaming sub-objects (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs as DIR/<name>.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    from fluidaudio_b200 import sharding, synth
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))

    if args.impl == "reference":
        if rank != 0:
            return 0
        threads = host_threads()
        steps = max(1, min(args.steps, 3))
        if args.workload == "mel":
            audio = synth.tone_noise_audio(MEL_SAMPLES)
            for _ in range(min(args.warmup, 1)):
                cpu_mel(audio[: 16000 * 120], threads)
            vals = [cpu_mel_arm(audio, threads, budget_s=8.0) for _ in range(steps)]
            v = float(np.mean([x[0] for x in vals])); dt = float(np.mean([x[1] for x in vals])); rep = vals[-1][2]
            v1, _ = cpu_mel(audio[: 16000 * 600], 1)
            vo, _ = cpu_mel(audio[: 16000 * 600], threads, 1, fast=False)
            line = {"impl": "reference", "metric": "audio-hours/s", "value": v, "unit": "audio-hours/s", "dtype": "f32",
                    "config": {"workload": "log-mel STFT, 1 h synthetic 16 kHz mono, 25 ms/10 ms frames, nFFT 512, 80 mels"},
                    "cpu_baseline": {"value": v, "unit": "audio-hours/s", "cores": threads, "kind": "port",
                                     "sample": f"the workload's hour of audio x {rep} per step, 30 s clips over {threads} threads: float32-FFT "
                                               "port of AudioMelSpectrogram.swift, SIMD across frames (oracle/oracle_mel_fast.cpp; no Swift "
                                               "toolchain, no Accelerate)",
                                     "single_thread_value": v1, "apple_m5_single_core_derived": 4.6,
                                     "parity_oracle_port_value": vo,
                                     "parity_oracle_port_note": "oracle_mel.cpp (float64 DFT rounded once, scalar), same threads, 600 s sample"}}
        else:
            emb, _ = synth.speaker_embeddings(CLUSTER_N, CLUSTER_D, CLUSTER_K, seed=42)
            rho, psi = synth.synthetic_plda(emb, CLUSTER_R)
            v, dt, kind, _ = cpu_cluster(emb, rho, psi)
            steps = 1
            line = {"impl": "reference", "metric": "embeddings/s", "value": v, "unit": "embeddings/s", "dtype": "f64",
                    "config": {"workload": "offline diarization backend: 10 000 x 256-d embeddings, AHC + VBx + assignment"},
                    "cpu_baseline": {"value": v, "unit": "embeddings/s", "cores": 1, "kind": kind,
                                     "sample": "the full 10 000 x 256 problem once; fastcluster is single-threaded as shipped"}}
        line.update({"n_gpus": args.gpus, "steps": steps, "warmup": args.warmup, "ms_per_step": dt * 1e3,
                     "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "data": "synthetic",
                     "e2e": {"value": v, "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})
        print(json.dumps(line))
        return 0

    from fluidaudio_b200 import _lib
    dist = sharding.init_distributed()
    if _lib.device_count() < 1:
        raise SystemExit("bench.py needs a B200: " + "no sm_100a device visible (there is no CPU fallback)")
    _lib.set_device(dist.local_rank)
    all_cpus = os.sched_getaffinity(0)
    numa = sharding.bind_to_gpu_numa(dist.local_rank)
    clocks = ClockSampler(dist.local_rank)

    got32 = None
    if args.workload == "mel":
        line, audio, got32, mel_out = bench_mel(args, dist, clocks)
        cluster_line, cluster_data = bench_cluster(args, dist)
        line["cluster"] = {k: cluster_line[k] for k in ("metric", "value", "unit", "ms_per_step", "e2e", "roofline", "stages_ms",
                                                         "gpu_launches", "config", "labels_equal_ref",
                                                         "labels_deterministic_all_ranks")}
        line["cluster"]["steps"] = args.steps
        if not args.only_main:
            line["c4"] = bench_c4(args, dist)
            line["c5"] = bench_c5(args, dist)
            if dist.is_root:
                line["streaming"] = bench_streaming(args)
    else:
        line, cluster_data = bench_cluster(args, dist)
        audio = mel_out = None
    line["clocks"] = clocks.summary()
    if args.dump_outputs and dist.is_root:
        dump_outputs(args.dump_outputs, mel_out, cluster_data[3])

    os.sched_setaffinity(0, all_cpus)      # the CPU baseline may use every host core again
    if dist.is_root and world == 1 and not args.no_cpu_baseline:
        threads = host_threads()
        if args.workload == "mel":
            from oracle import oracle as O
            v, dt, rep = cpu_mel_arm(audio, threads, budget_s=8.0)
            v1, _ = cpu_mel(audio[: 16000 * 600], 1)
            vo, _ = cpu_mel(audio[: 16000 * 600], threads, 1, fast=False)
            line["cpu_baseline"] = {"value": v, "unit": "audio-hours/s", "cores": threads, "kind": "port",
                                    "sample": f"the workload's hour of audio x {rep}, 30 s clips over {threads} host threads, {dt:.2f} s wall: "
                                              "float32-FFT port of AudioMelSpectrogram.swift, SIMD across frames (oracle/oracle_mel_fast.cpp)",
                                    "single_thread_value": v1, "apple_m5_single_core_derived": 4.6,
                                    "parity_oracle_port_value": vo}
            # the CPU arms double as checkers of the GPU output (first minute): the parity oracle and the float32 port
            cfg = O.mel_config(n_mels=N_MELS)
            ref, rml, _ = O.mel_flat_transposed(cfg, audio[:960000])
            fast, _ = O.mel_fast_flat_transposed(cfg, audio[:960000], 0.0)
            line["parity"]["max_abs_vs_oracle_first_minute"] = float(np.abs(got32[:rml - 3] - ref[:rml - 3]).max())
            line["parity"]["max_abs_vs_cpu_float32_port_first_minute"] = float(np.abs(got32[:rml - 3] - fast[:rml - 3]).max())
            emb, rho, psi, res = cluster_data
            cv, cdt, kind, ores = cpu_cluster(emb, rho, psi)
            line["cluster"]["cpu_baseline"] = {"value": cv, "unit": "embeddings/s", "cores": 1, "kind": kind,
                                               "sample": f"the full 10 000 x 256 problem once, {cdt:.1f} s "
                                                         "(fastcluster is single-threaded as shipped)"}
            line["cluster"]["labels_equal_cpu"] = bool(np.array_equal(res.labels, ores.labels))
        else:
            emb, rho, psi, res = cluster_data
            cv, cdt, kind, ores = cpu_cluster(emb, rho, psi)
            line["cpu_baseline"] = {"value": cv, "unit": "embeddings/s", "cores": 1, "kind": kind,
                                    "sample": f"the full 10 000 x 256 problem once, {cdt:.1f} s"}
            line["labels_equal_cpu"] = bool(np.array_equal(res.labels, ores.labels))

    line["host_binding"] = numa
    line.update({"n_gpus": dist.world, "steps": args.steps, "warmup": args.warmup, "higher_is_better": True,
                 "scaling": "weak", "vs_baseline": None, "data": "synthetic"})
    if dist.is_root:
        print(json.dumps(line))
    sharding.finalize(dist)
    return 0


if __name__ == "__main__":
    sys.exit(main())
