"""ORACLE — TEST INFRASTRUCTURE ONLY.  Not part of the shipped product path.

ctypes front-end to ``liboracle.so`` (our CPU restatement, ``oracle_*.cpp``) and, when present, to
``_ref/liboracle_fc.so`` (the unmodified reference ``FastClusterWrapper.cpp`` compiled by ``make ref``); where that was
not built, the restatement stands in for it only where it reproduces the reference's results recorded in
``tests/golden/ref_linkage.json``.
Importers allowed: ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s cpu_baseline / ``--impl reference``.
The product package ``fluidaudio_b200`` must never import this module (tests enforce it).

Pipeline glue restated here (pure Python, O(N)):
  * ``ahc_cluster``      AHCClustering.cluster            AHCClustering.swift:20-67
  * ``vbx_refine``       VBxClustering.refine             VBxClustering.swift:41-165
  * ``diarize_cluster``  OfflineDiarizerManager.cluster   OfflineDiarizerManager.swift:270-384 (+591-611)
"""
from __future__ import annotations

import ctypes as C
import hashlib
import json
import os
import subprocess
from dataclasses import dataclass

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = os.path.join(_HERE, "liboracle.so")
_REF = os.path.join(_HERE, "_ref", "liboracle_fc.so")
_RECORDED = os.path.join(os.path.dirname(_HERE), "tests", "golden", "ref_linkage.json")
_REFERENCE_ROOT = "/root/reference"

_f32p = np.ctypeslib.ndpointer(np.float32, flags="C_CONTIGUOUS")
_f64p = np.ctypeslib.ndpointer(np.float64, flags="C_CONTIGUOUS")
_i32p = np.ctypeslib.ndpointer(np.int32, flags="C_CONTIGUOUS")


def build(force: bool = False) -> None:
    """Compile liboracle.so (always possible) and _ref/liboracle_fc.so (only where /root/reference exists)."""
    srcs = [os.path.join(_HERE, f) for f in ("oracle_mel.cpp", "oracle_cluster.cpp", "oracle_adapters.cpp",
                                             "oracle_mel_fast.cpp")]
    stale = force or not os.path.exists(_LIB) or any(os.path.getmtime(s) > os.path.getmtime(_LIB) for s in srcs)
    if stale:
        subprocess.check_call(["make", "-s", "-C", _HERE, "-B", "all"])
    ref_src = os.path.join(_REFERENCE_ROOT, "Sources/FastClusterWrapper/FastClusterWrapper.cpp")
    if os.path.exists(ref_src) and (force or not os.path.exists(_REF)):
        subprocess.check_call(["make", "-s", "-C", _HERE, "-B", "ref"])


class MelConfig(C.Structure):
    _fields_ = [
        ("sample_rate", C.c_int32), ("n_mels", C.c_int32), ("n_fft", C.c_int32), ("hop_length", C.c_int32),
        ("win_length", C.c_int32), ("preemph", C.c_float), ("pad_to", C.c_int32), ("log_floor", C.c_float),
        ("log_floor_mode", C.c_int32), ("window_periodic", C.c_int32), ("precision", C.c_int32),
    ]


class VbxConfig(C.Structure):
    _fields_ = [("Fa", C.c_double), ("Fb", C.c_double), ("max_iterations", C.c_int32), ("epsilon", C.c_double),
                ("init_smoothing", C.c_double)]


_lib = None
_ref = None
_recorded = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB):
            build()
        L = C.CDLL(_LIB)
        L.oracle_mel_hann.argtypes = [C.c_int32, C.c_int32, _f32p]
        L.oracle_mel_filterbank.argtypes = [C.c_int32, C.c_int32, C.c_int32, _f32p]
        L.oracle_mel_frame_count.argtypes = [C.POINTER(MelConfig), C.c_int64, C.c_int32, C.c_int64]
        L.oracle_mel_frame_count.restype = C.c_int64
        for name in ("oracle_mel_compute_flat_transposed",):
            f = getattr(L, name)
            f.argtypes = [C.POINTER(MelConfig), C.c_void_p, C.c_int64, C.c_float, C.c_int32, C.c_int64,
                          C.c_void_p, C.c_int64, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
            f.restype = C.c_int64
        L.oracle_mel_compute_flat.argtypes = [C.POINTER(MelConfig), C.c_void_p, C.c_int64, C.c_float, C.c_void_p,
                                              C.c_int64, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
        L.oracle_mel_compute_flat.restype = C.c_int64
        L.oracle_mel_compute_legacy.argtypes = [C.POINTER(MelConfig), C.c_void_p, C.c_int64, C.c_void_p, C.c_int64,
                                                C.POINTER(C.c_int64)]
        L.oracle_mel_compute_legacy.restype = C.c_int64
        L.oracle_l2_normalize_rows.argtypes = [_f64p, C.c_int64, C.c_int64, _f64p]
        L.oracle_centroid_linkage.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p, C.c_uint64]
        L.oracle_centroid_linkage.restype = C.c_int32
        L.oracle_dendrogram_cut.argtypes = [_f64p, C.c_int64, C.c_double, _i32p]
        L.oracle_vbx_refine.argtypes = [_f64p, C.c_int64, C.c_int64, _f64p, C.c_int64, C.c_void_p,
                                        C.POINTER(VbxConfig), C.c_int32, _f64p, _f64p, _f64p, _i32p]
        L.oracle_vbx_refine.restype = C.c_int32
        L.oracle_compute_centroids.argtypes = [_f64p, C.c_int64, C.c_int64, _f64p, _f64p, C.c_int32, _f64p, _i32p]
        L.oracle_compute_centroids.restype = C.c_int32
        L.oracle_centroids_from_clusters.argtypes = [_f64p, C.c_int64, C.c_int64, _i32p, _f64p, C.c_int32]
        L.oracle_centroids_from_clusters.restype = C.c_int32
        L.oracle_assign_embeddings.argtypes = [_f64p, C.c_int64, C.c_int64, _f64p, C.c_int32, _i32p, C.c_void_p]
        L.oracle_hungarian_solve.argtypes = [np.ctypeslib.ndpointer(np.int64, flags="C_CONTIGUOUS"), C.c_int32, _i32p]
        L.oracle_max_score_assignment.argtypes = [_f64p, C.c_int32, C.c_int32, _i32p]
        L.oracle_constrained_assign.argtypes = [_f64p, C.c_int64, C.c_int32, _i32p, _i32p]
        L.oracle_build_chunk_assignments.argtypes = [_i32p, _i32p, _i32p, C.c_int64, C.c_int32, C.c_int32, C.c_int32, _i32p]
        L.oracle_linear_resample.argtypes = [_f32p, C.c_int64, C.c_int32, C.c_double, C.c_double, C.c_void_p]
        L.oracle_linear_resample.restype = C.c_int64
        L.oracle_normalize_per_feature.argtypes = [_f32p, C.c_int64, C.c_int32, C.c_int64]
        L.oracle_kmeans.argtypes = [_f64p, C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_uint64, _i32p, _f64p,
                                    C.POINTER(C.c_int32)]
        L.oracle_kmeans.restype = C.c_int32
        L.oracle_kmeans_ninit.argtypes = [_f64p, C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_uint64, _i32p,
                                          _f64p, C.POINTER(C.c_int32)]
        L.oracle_kmeans_ninit.restype = C.c_int32
        L.oracle_speaker_constraints.argtypes = [C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.POINTER(C.c_int64)]
        L.oracle_speaker_constraints.restype = None
        L.oracle_lseend_scale_cmn.argtypes = [_f32p, C.c_int64, C.c_int32, _f32p, C.POINTER(C.c_int64)]
        L.oracle_lseend_scale_cmn.restype = None
        L.oracle_transpose_tm.argtypes = [_f32p, C.c_int64, C.c_int32, _f32p]
        _lib = L
    return _lib


def ref_available() -> bool:
    return os.path.exists(_REF)


def ref():
    """The compiled, unmodified reference FastClusterWrapper (None if it was never built here)."""
    global _ref
    if _ref is None and os.path.exists(_REF):
        R = C.CDLL(_REF)
        R.fastcluster_compute_centroid_linkage.argtypes = [C.c_void_p, C.c_size_t, C.c_size_t, C.c_void_p, C.c_size_t]
        R.fastcluster_compute_centroid_linkage.restype = C.c_int
        _ref = R
    return _ref


# ------------------------------------------------------------------------------------------------ mel
def mel_config(sample_rate=16000, n_mels=128, n_fft=512, hop_length=160, win_length=400, preemph=0.97, pad_to=0,
               log_floor=2.0 ** -24, log_floor_mode=0, window_periodic=False, precision=0) -> MelConfig:
    return MelConfig(sample_rate, n_mels, n_fft, hop_length, win_length, preemph, pad_to, log_floor,
                     log_floor_mode, int(window_periodic), precision)


def hann_window(length=400, periodic=False) -> np.ndarray:
    out = np.zeros(length, np.float32)
    lib().oracle_mel_hann(length, int(periodic), out)
    return out


def mel_filterbank(n_fft=512, n_mels=128, sample_rate=16000) -> np.ndarray:
    out = np.zeros((n_mels, n_fft // 2 + 1), np.float32)
    lib().oracle_mel_filterbank(n_fft, n_mels, sample_rate, out)
    return out


def mel_frame_count(cfg: MelConfig, n: int, mode: int = 0, expected: int = -1) -> int:
    return int(lib().oracle_mel_frame_count(C.byref(cfg), n, mode, expected))


def mel_flat_transposed(cfg: MelConfig, audio: np.ndarray, last=0.0, padding_mode=0, expected_frames=None):
    """computeFlatTransposed: returns (mel [Tp x nMels] float32, melLength, numFrames)."""
    audio = np.ascontiguousarray(audio, np.float32)
    exp = -1 if expected_frames is None else int(expected_frames)
    ml, nf = C.c_int64(), C.c_int64()
    need = lib().oracle_mel_compute_flat_transposed(C.byref(cfg), audio.ctypes.data, audio.size, last, padding_mode,
                                                    exp, None, 0, C.byref(ml), C.byref(nf))
    out = np.zeros(need, np.float32)
    lib().oracle_mel_compute_flat_transposed(C.byref(cfg), audio.ctypes.data, audio.size, last, padding_mode, exp,
                                             out.ctypes.data, need, C.byref(ml), C.byref(nf))
    if ml.value == 0:
        return out, 0, 1
    return out.reshape(nf.value, cfg.n_mels), ml.value, nf.value


def mel_fast_flat_transposed(cfg: MelConfig, audio: np.ndarray, last=0.0):
    """The TIMED CPU arm (oracle_mel_fast.cpp): float32 FFT, SIMD across frames; .center, pad_to 1, nFFT 512."""
    audio = np.ascontiguousarray(audio, np.float32)
    L = lib()
    L.oracle_mel_fast_flat_transposed.restype = C.c_int64
    L.oracle_mel_fast_flat_transposed.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_float, C.c_void_p, C.c_int64,
                                                  C.POINTER(C.c_int64)]
    ml = C.c_int64()
    need = L.oracle_mel_fast_flat_transposed(C.byref(cfg), audio.ctypes.data, audio.size, float(last), None, 0, C.byref(ml))
    out = np.zeros(need, np.float32)
    L.oracle_mel_fast_flat_transposed(C.byref(cfg), audio.ctypes.data, audio.size, float(last), out.ctypes.data, need, C.byref(ml))
    return out.reshape(ml.value, cfg.n_mels), int(ml.value)


def mel_flat(cfg: MelConfig, audio: np.ndarray, last=0.0):
    """computeFlat: returns (mel [nMels x Tp], melLength, numFrames)."""
    audio = np.ascontiguousarray(audio, np.float32)
    ml, nf = C.c_int64(), C.c_int64()
    need = lib().oracle_mel_compute_flat(C.byref(cfg), audio.ctypes.data, audio.size, last, None, 0, C.byref(ml),
                                         C.byref(nf))
    out = np.zeros(need, np.float32)
    lib().oracle_mel_compute_flat(C.byref(cfg), audio.ctypes.data, audio.size, last, out.ctypes.data, need,
                                  C.byref(ml), C.byref(nf))
    if ml.value == 0:
        return out, 0, 1
    return out.reshape(cfg.n_mels, nf.value), ml.value, nf.value


def mel_legacy(cfg: MelConfig, audio: np.ndarray):
    """compute(audio:): returns (mel [nMels x T], melLength)."""
    audio = np.ascontiguousarray(audio, np.float32)
    ml = C.c_int64()
    need = lib().oracle_mel_compute_legacy(C.byref(cfg), audio.ctypes.data, audio.size, None, 0, C.byref(ml))
    if need <= 0:
        return np.zeros((0,), np.float32), 0
    out = np.zeros(need, np.float32)
    lib().oracle_mel_compute_legacy(C.byref(cfg), audio.ctypes.data, audio.size, out.ctypes.data, need, C.byref(ml))
    return out.reshape(cfg.n_mels, ml.value), ml.value


def normalize_per_feature(x: np.ndarray, valid_frames: int) -> np.ndarray:
    y = np.ascontiguousarray(x, np.float32).copy()
    lib().oracle_normalize_per_feature(y, y.shape[0], y.shape[1], valid_frames)
    return y


def unified_mel_features(window: np.ndarray, valid_count: int, n_mels: int = 128, hop: int = 160):
    """UnifiedMelExtractor.features(window:validCount:) (UnifiedMelExtractor.swift:52-86): center-padded log-mel with
    expectedFrameCount = windowSamples / hop + 1, NeMo per-feature normalisation over validCount / hop frames, packed as
    [nMels x totalFrames].  Returns (mel [n_mels x T], valid_frames)."""
    window = np.ascontiguousarray(window, np.float32)
    total = window.size // hop + 1
    cfg = mel_config(n_mels=n_mels)
    flat, _, _ = mel_flat_transposed(cfg, window, 0.0, 0, expected_frames=total)
    valid = min(int(valid_count) // hop, total)
    norm = normalize_per_feature(flat[:total], valid)
    return np.ascontiguousarray(norm.T), valid


def lseend_config(n_mels: int = 23, n_fft: int = 512, hop_length: int = 160, win_length: int = 400, sample_rate: int = 16000):
    """The AudioMelSpectrogram LSEENDPreprocessor builds (LSEENDPreprocessor.swift:70-81)."""
    return mel_config(sample_rate=sample_rate, n_mels=n_mels, n_fft=n_fft, hop_length=hop_length, win_length=win_length,
                      preemph=0.0, pad_to=0, log_floor=1e-10, log_floor_mode=1, window_periodic=True)


def lseend_features(cfg: MelConfig, chunk: np.ndarray, cmn_mean: np.ndarray, cmn_count: int):
    """LSEENDPreprocessor.processAudioQueue (:249-283): .prePadded log-mel, log10 scaling, cumulative mean
    normalisation.  Returns (features [T x nMels], cmn_mean', cmn_count')."""
    flat, ml, _ = mel_flat_transposed(cfg, np.ascontiguousarray(chunk, np.float32), 0.0, 1, None)
    x = np.ascontiguousarray(flat[:ml], np.float32).copy()
    mean = np.ascontiguousarray(cmn_mean, np.float32).copy()
    cnt = C.c_int64(int(cmn_count))
    lib().oracle_lseend_scale_cmn(x, x.shape[0], x.shape[1], mean, C.byref(cnt))
    return x, mean, cnt.value


def linear_resample(planar: np.ndarray, in_rate: float, out_rate: float) -> np.ndarray:
    """planar: [channels x frames] float32."""
    planar = np.ascontiguousarray(planar, np.float32)
    ch, frames = planar.shape
    n = lib().oracle_linear_resample(planar, frames, ch, in_rate, out_rate, None)
    out = np.zeros(n, np.float32)
    lib().oracle_linear_resample(planar, frames, ch, in_rate, out_rate, out.ctypes.data)
    return out


# ---- AudioConverter stage (R1).  The reference's one- and two-channel path is Apple's closed AVAudioConverter
# (AudioConverter.swift:299-375): PARITY UNPINNED for sample values.  What is restated here is the replacement filter the
# library documents (fluidaudio_b200/csrc/resample_plan.h): Kaiser-windowed sinc, evaluated in float64, so that the GPU
# kernel can be checked against its own specification; the reference-held facts (identity at the target rate :66-68,
# output length rule :417-418 and +-1 % AudioConverterTests.swift:129-176, mean mixdown :401-409) are tested directly.
SINC_ROLLOFF, SINC_ZEROS, SINC_BETA = 0.94, 24, 12.0


def resample_output_count(frames: int, in_rate: float, out_rate: float) -> int:
    return int(frames) if in_rate == out_rate else int(float(frames) / (in_rate / out_rate))


def rational_ratio(in_rate: float, out_rate: float):
    """out/in = L/M in lowest terms, reduced as the library does (resample_kernels.cu rational_ratio): integer rates as
    they are, otherwise both rates on a 1/1000 Hz grid (rounded to the nearest grid point), then divided by their gcd."""
    from math import floor, gcd
    whole = lambda r: abs(r - round(r)) <= 1e-9
    scale = 1 if whole(in_rate) and whole(out_rate) else 1000
    a, b = int(floor(out_rate * scale + 0.5)), int(floor(in_rate * scale + 0.5))
    g = gcd(a, b)
    return a // g, b // g


def sinc_design(in_rate: float, out_rate: float):
    """Returns (L, M, half, fc): out/in = L/M, half = taps / 2, fc relative to the input Nyquist."""
    L, M = rational_ratio(in_rate, out_rate)
    lower = min(1.0, L / M)
    return L, M, int(np.ceil(SINC_ZEROS / lower)), lower * SINC_ROLLOFF


def _sinc_kernel(t: np.ndarray, half: int, fc: float) -> np.ndarray:
    u = np.clip(1.0 - (t / half) ** 2, 0.0, None)
    g = fc * np.sinc(fc * t) * np.i0(SINC_BETA * np.sqrt(u)) / np.i0(SINC_BETA)
    return np.where(np.abs(t) < half, g, 0.0)


def mixdown(pcm: np.ndarray) -> np.ndarray:
    """[channels x frames] float32 / int16 -> mono float32: sequential float32 sum, times float32(1/channels)
    (AudioConverter.swift:401-409); int16 widened as v / 32768."""
    x = np.asarray(pcm)
    if x.ndim == 1:
        x = x[None]
    if x.dtype == np.int16:
        x = x.astype(np.float32) * np.float32(1.0 / 32768.0)
    x = x.astype(np.float32)
    s = np.zeros(x.shape[1], np.float32)
    for c in range(x.shape[0]):
        s = (s + x[c]).astype(np.float32)
    return s if x.shape[0] == 1 else (s * np.float32(1.0 / np.float32(x.shape[0]))).astype(np.float32)


def sinc_resample(mono: np.ndarray, in_rate: float, out_rate: float, first: int = 0, count=None) -> np.ndarray:
    """float64 evaluation of the documented polyphase filter on a mono float32 signal (rows normalised to unit DC gain
    exactly as the library's float32 table is, so the only difference left is float32 rounding of taps and sums).
    Evaluates outputs [first, first + count) of the whole signal's resampling (default: all of them), each at its exact
    phase (i * M) mod L, so a window at the far end of a long signal costs what a window at its start does."""
    x = np.asarray(mono, np.float32).astype(np.float64)
    n = x.size
    total = resample_output_count(n, in_rate, out_rate)
    count = total - first if count is None else int(count)
    if first < 0 or count < 0 or first + count > total:
        raise ValueError(f"outputs [{first}, {first + count}) outside [0, {total})")
    if in_rate == out_rate:
        return x[first:first + count].astype(np.float32)
    L, M, half, fc = sinc_design(in_rate, out_rate)
    k = np.arange(-half + 1, half + 1)
    rows_of = None
    if L <= 4096:                   # few distinct phases: one normalised row per phase, shared by the outputs
        table = _sinc_kernel(k[None, :] - np.arange(L)[:, None] / L, half, fc)
        table /= table.sum(axis=1, keepdims=True)
        rows_of = lambda ph: table[ph]
    out = np.zeros(count)
    block = 4096
    for s in range(0, count, block):
        i = np.arange(first + s, first + min(s + block, count), dtype=np.int64)
        num = i * M                 # < 2^63 for any signal a test can hold
        n0, ph = num // L, num % L
        if rows_of is not None:
            rows = rows_of(ph)
        else:
            rows = _sinc_kernel(k[None, :] - ph[:, None] / L, half, fc)
            rows /= rows.sum(axis=1, keepdims=True)
        idx = n0[:, None] + k[None, :]
        xs = np.where((idx >= 0) & (idx < n), x[np.clip(idx, 0, max(n - 1, 0))], 0.0)
        out[s:s + i.size] = (xs * rows).sum(axis=1)
    return out.astype(np.float32)


# ------------------------------------------------------------------------------------------------ clustering
def l2_normalize_rows(x: np.ndarray) -> np.ndarray:
    x = np.ascontiguousarray(x, np.float64)
    out = np.zeros_like(x)
    lib().oracle_l2_normalize_rows(x, x.shape[0], x.shape[1], out)
    return out


def _linkage_key(x: np.ndarray) -> str:
    return hashlib.sha256(np.asarray(x.shape, np.int64).tobytes() + x.tobytes()).hexdigest()[:32]


def _linkage_record(status: int, z: np.ndarray) -> dict:
    """What is kept of a reference result: its status and, when it succeeded, the SHA-256 of the dendrogram bytes."""
    return {"status": int(status), "z_sha256": hashlib.sha256(z.tobytes()).hexdigest() if status == 0 else None}


def reference_linkage(x: np.ndarray):
    """The reference's (status, Z) for x.  Computed by the compiled reference where `make ref` built it; elsewhere the
    restatement's result, accepted only if it reproduces the reference's status and dendrogram bytes (SHA-256) recorded for
    the same input in tests/golden/ref_linkage.json (how to record new inputs: tests/golden/make_golden.py).  With
    FA_ORACLE_RECORD_REF=<dir> every call to the compiled reference also stores its record under <dir>."""
    global _recorded
    x = np.ascontiguousarray(x, np.float64)
    key = _linkage_key(x)
    if ref() is None:
        if _recorded is None:
            with open(_RECORDED) as f:
                _recorded = json.load(f)
        if key not in _recorded:
            raise LookupError(f"no recorded reference result for this {x.shape} input (key {key}): record it with the "
                              "compiled reference (tests/golden/make_golden.py)")
        st, z = centroid_linkage(x)
        if _linkage_record(st, z) != _recorded[key]:
            raise AssertionError(f"the restatement differs from the reference's recorded result for this {x.shape} input "
                                 f"(key {key})")
        return st, z
    n, d = x.shape
    z = np.zeros((max(n - 1, 0), 4), np.float64)
    zp = z.ctypes.data if z.size else C.cast(C.create_string_buffer(8), C.c_void_p).value
    st = int(ref().fastcluster_compute_centroid_linkage(x.ctypes.data, n, d, zp, z.size))
    out_dir = os.environ.get("FA_ORACLE_RECORD_REF")
    if out_dir:
        os.makedirs(out_dir, exist_ok=True)
        with open(os.path.join(out_dir, key + ".json"), "w") as f:
            json.dump(_linkage_record(st, z), f)
    return st, z


def centroid_linkage(x: np.ndarray, use_ref: bool = False):
    """Returns (status, Z [(N-1) x 4]).  use_ref=True gives the reference's result (reference_linkage) instead of the
    restatement's."""
    x = np.ascontiguousarray(x, np.float64)
    if use_ref:
        return reference_linkage(x)
    n, d = x.shape
    z = np.zeros((max(n - 1, 0), 4), np.float64)
    zp = z.ctypes.data if z.size else C.cast(C.create_string_buffer(8), C.c_void_p).value
    st = lib().oracle_centroid_linkage(x.ctypes.data, n, d, zp, z.size)
    return int(st), z


def dendrogram_cut(z: np.ndarray, count: int, threshold: float) -> np.ndarray:
    labels = np.zeros(count, np.int32)
    zz = np.ascontiguousarray(z, np.float64).reshape(-1)
    if zz.size == 0:
        zz = np.zeros(4, np.float64)
    lib().oracle_dendrogram_cut(zz, count, threshold, labels)
    return labels


def ahc_cluster(features: np.ndarray, threshold: float, use_ref: bool = False) -> np.ndarray:
    """AHCClustering.cluster (AHCClustering.swift:20-67) incl. guards and the FFI-failure fallback."""
    features = np.asarray(features, np.float64)
    count = features.shape[0]
    if count == 0:
        return np.zeros(0, np.int32)
    if features.ndim < 2 or features.shape[1] == 0:
        return np.zeros(count, np.int32)
    if count == 1:
        return np.zeros(1, np.int32)
    normalized = l2_normalize_rows(features)
    status, z = centroid_linkage(normalized, use_ref=use_ref)
    if status != 0:
        return np.arange(count, dtype=np.int32)
    return dendrogram_cut(z, count, threshold)


@dataclass
class VBxOutput:
    gamma: np.ndarray
    pi: np.ndarray
    hard: np.ndarray
    num_clusters: int
    elbos: np.ndarray


def vbx_refine(rho: np.ndarray, psi: np.ndarray, initial: np.ndarray, Fa=0.07, Fb=0.8, max_iterations=20,
               epsilon=1e-4, init_smoothing=7.0) -> VBxOutput:
    rho = np.ascontiguousarray(rho, np.float64)
    T = rho.shape[0]
    if T == 0 or rho.ndim < 2 or rho.shape[1] == 0:
        return VBxOutput(np.zeros((0, 0)), np.zeros(0), np.zeros(0, np.int32), 0, np.zeros(0))
    D = rho.shape[1]
    psi = np.ascontiguousarray(psi, np.float64)
    initial = np.ascontiguousarray(initial, np.int32)
    S = max(1, len(set(initial.tolist())))
    gamma = np.zeros((T, S), np.float64)
    pi = np.zeros(S, np.float64)
    elbos = np.zeros(max(max_iterations, 1), np.float64)
    hard = np.zeros(T, np.int32)
    cfg = VbxConfig(Fa, Fb, max_iterations, epsilon, init_smoothing)
    init_ptr = initial.ctypes.data if initial.size else None
    iters = lib().oracle_vbx_refine(rho, T, D, psi if psi.size else np.zeros(1), psi.size, init_ptr, C.byref(cfg), S,
                                    gamma, pi, elbos, hard)
    return VBxOutput(gamma, pi, hard, S, elbos[:iters].copy())


def compute_centroids(train: np.ndarray, vbx: VBxOutput, initial: np.ndarray) -> np.ndarray:
    """computeCentroids (OfflineDiarizerManager.swift:613-691) with the from-clusters fallback (:693-746)."""
    train = np.ascontiguousarray(train, np.float64)
    T, dim = train.shape
    if vbx.gamma.size and vbx.pi.size and np.any(vbx.pi > 1e-7):
        S = vbx.pi.size
        cents = np.zeros((S, dim), np.float64)
        who = np.zeros(S, np.int32)
        limit = min(vbx.gamma.shape[0], T)
        K = lib().oracle_compute_centroids(train[:limit].copy(), limit, dim,
                                           np.ascontiguousarray(vbx.gamma[:limit]), vbx.pi, S, cents, who)
        return cents[:K].copy()
    initial = np.ascontiguousarray(initial, np.int32)
    if T == 0 or initial.size != T:
        return np.zeros((0, dim))
    cap = len(set(initial.tolist()))
    cents = np.zeros((cap, dim), np.float64)
    K = lib().oracle_centroids_from_clusters(train, T, dim, initial, cents, cap)
    return cents[:K].copy()


def assign_embeddings(emb: np.ndarray, centroids: np.ndarray, want_scores=False):
    emb = np.ascontiguousarray(emb, np.float64)
    centroids = np.ascontiguousarray(centroids, np.float64)
    N, dim = emb.shape
    K = centroids.shape[0]
    labels = np.zeros(N, np.int32)
    scores = np.zeros((N, max(K, 1)), np.float64) if want_scores else None
    lib().oracle_assign_embeddings(emb, N, dim, centroids if K else np.zeros((1, dim)), K, labels,
                                   scores.ctypes.data if want_scores else None)
    return (labels, scores) if want_scores else labels


def hungarian_solve(cost: np.ndarray) -> np.ndarray:
    cost = np.ascontiguousarray(cost, np.int64)
    n = cost.shape[0] if cost.ndim == 2 else int(round(cost.size ** 0.5))
    out = np.zeros(max(n, 1), np.int32)
    if n:
        lib().oracle_hungarian_solve(cost.reshape(-1), n, out)
    return out[:n]


def max_score_assignment(scores) -> np.ndarray:
    scores = np.ascontiguousarray(scores, np.float64)
    rows = scores.shape[0]
    cols = scores.shape[1] if scores.ndim == 2 else 0
    out = np.zeros(max(rows, 1), np.int32)
    if rows:
        lib().oracle_max_score_assignment(scores.reshape(-1) if scores.size else np.zeros(1), rows, cols, out)
    return out[:rows]


def constrained_assign(scores, chunk_indices) -> np.ndarray:
    scores = np.ascontiguousarray(scores, np.float64)
    chunk = np.ascontiguousarray(chunk_indices, np.int32)
    N = chunk.size
    K = scores.shape[1] if scores.ndim == 2 else 0
    out = np.zeros(max(N, 1), np.int32)
    if N:
        lib().oracle_constrained_assign(scores.reshape(-1) if scores.size else np.zeros(1), N, K, chunk, out)
    return out[:N]


def build_chunk_assignments(chunk, speaker, assignments, num_chunks, num_speakers, cluster_count) -> np.ndarray:
    chunk = np.ascontiguousarray(chunk, np.int32)
    speaker = np.ascontiguousarray(speaker, np.int32)
    assignments = np.ascontiguousarray(assignments, np.int32)
    m = np.zeros((num_chunks, num_speakers), np.int32)
    lib().oracle_build_chunk_assignments(chunk, speaker, assignments, chunk.size, num_chunks, num_speakers, cluster_count,
                                         m.reshape(-1))
    return m


@dataclass
class ClusterResult:
    labels: np.ndarray          # final assignment for all N embeddings (P3)
    initial: np.ndarray         # AHC labels of the training subset (A1)
    vbx: VBxOutput
    centroids: np.ndarray
    training_indices: np.ndarray
    was_adjusted: bool = False  # VBxOutput.wasAdjusted (K-Means replaced the VBx clusters)
    detected_clusters: int = 0  # VBxOutput.assignedClusterCount


class _OracleSegment(C.Structure):
    _fields_ = [("cluster", C.c_int32), ("start", C.c_float), ("end", C.c_float), ("quality", C.c_float)]


class _OracleReconstructConfig(C.Structure):
    _fields_ = [("frame_duration", C.c_double), ("window_duration", C.c_double), ("min_gap_duration", C.c_double),
                ("seg_min_duration_off", C.c_double), ("seg_min_duration_on", C.c_double),
                ("min_segment_duration", C.c_double), ("exclusive_segments", C.c_int32)]


def build_segments(speaker_weights, hard_clusters, centroid_count, frame_duration, chunk_offsets=None, window_duration=10.0,
                   min_gap_duration=0.1, seg_min_duration_off=0.0, seg_min_duration_on=0.0, min_segment_duration=1.0,
                   exclusive_segments=True):
    """OfflineReconstruction.buildSegments (:24-253) -> list of (cluster, start, end, quality)."""
    w = np.ascontiguousarray(speaker_weights, np.float32)
    chunks, frames, speakers = w.shape if w.ndim == 3 else (0, 0, 0)
    hard = np.ascontiguousarray(hard_clusters, np.int32).reshape(-1, max(speakers, 1)) if np.size(hard_clusters) else \
        np.zeros((0, max(speakers, 1)), np.int32)
    offs = np.ascontiguousarray(chunk_offsets if chunk_offsets is not None else [], np.float64)
    cfg = _OracleReconstructConfig(frame_duration, window_duration, min_gap_duration, seg_min_duration_off,
                                   seg_min_duration_on, min_segment_duration, int(exclusive_segments))
    L = lib()
    L.oracle_build_segments.restype = C.c_int32
    L.oracle_build_segments.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p,
                                        C.c_int32, C.c_int32, C.POINTER(_OracleReconstructConfig), C.c_void_p, C.c_int32]
    cap = max(16, chunks * max(speakers, 1) * 4 + 16)
    while True:
        buf = (_OracleSegment * cap)()
        n = L.oracle_build_segments(w.ctypes.data if w.size else None, chunks, frames, speakers,
                                    offs.ctypes.data if offs.size else None, offs.size,
                                    hard.ctypes.data if hard.size else None, hard.shape[0], centroid_count, C.byref(cfg), buf, cap)
        if n <= cap:
            return [(buf[i].cluster, buf[i].start, buf[i].end, buf[i].quality) for i in range(n)]
        cap = n


def build_speaker_database(seg_clusters, centroids):
    """OfflineReconstruction.buildSpeakerDatabase (:296-357) -> (database float32 [K x dim], segment counts [K])."""
    cl = np.ascontiguousarray(seg_clusters, np.int32)
    cen = np.ascontiguousarray(centroids, np.float64)
    K, dim = cen.shape
    db = np.zeros((K, dim), np.float32)
    counts = np.zeros(K, np.int32)
    L = lib()
    L.oracle_build_speaker_database.restype = None
    L.oracle_build_speaker_database.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]
    L.oracle_build_speaker_database(cl.ctypes.data if cl.size else None, cl.size, cen.ctypes.data, K, dim, db.ctypes.data,
                                    counts.ctypes.data)
    return db, counts


def kmeans(emb: np.ndarray, num_clusters: int, max_iterations: int = 300, seed: int = 0):
    """KMeansClustering.clusterWithCentroids (:39-92): (labels, centroids, loop iterations)."""
    emb = np.ascontiguousarray(emb, np.float64)
    n, d = emb.shape
    labels = np.zeros(n, np.int32)
    cents = np.zeros((max(1, min(num_clusters, n)), d), np.float64)
    it = C.c_int32()
    rows = lib().oracle_kmeans(emb, n, d, num_clusters, max_iterations, seed, labels, cents, C.byref(it))
    return labels, cents[:rows].copy(), it.value


def kmeans_ninit(emb: np.ndarray, num_clusters: int, max_iterations: int = 300, n_init: int = 10, base_seed: int = 0):
    """KMeansClustering.clusterWithCentroidsNInit (:99-130): (labels, centroids, winning init)."""
    emb = np.ascontiguousarray(emb, np.float64)
    n, d = emb.shape
    labels = np.zeros(n, np.int32)
    cents = np.zeros((max(1, min(num_clusters, n)), d), np.float64)
    best = C.c_int32()
    rows = lib().oracle_kmeans_ninit(emb, n, d, num_clusters, max_iterations, n_init, base_seed, labels, cents,
                                     C.byref(best))
    return labels, cents[:rows].copy(), best.value


def speaker_constraints(num_embeddings: int, num_speakers=None, min_speakers=None, max_speakers=None):
    """SpeakerCountConstraints.resolve (:27-71): (min, max)."""
    opt = lambda v: -2 ** 63 if v is None else int(v)
    out = (C.c_int64 * 2)()
    lib().oracle_speaker_constraints(num_embeddings, opt(num_speakers), opt(min_speakers), opt(max_speakers), out)
    return int(out[0]), int(out[1])


def diarize_cluster(emb256: np.ndarray, rho128: np.ndarray, psi: np.ndarray, threshold=0.6, Fa=0.07, Fb=0.8,
                    max_iterations=20, epsilon=1e-4, use_ref: bool = False, chunk_indices=None, num_speakers=None,
                    min_speakers=None, max_speakers=None) -> ClusterResult:
    """OfflineDiarizerManager.cluster(_:) lines 286-375.  chunk_indices=None -> plain argmax (:371-374); otherwise
    the reference's default constrained assignment (:357-369) whenever more than one centroid exists and the speaker
    count was not forced.  num/min/max_speakers: VBxClustering.refineWithConstraints (:685-733)."""
    emb32 = np.ascontiguousarray(emb256, np.float32)
    feats = emb32.astype(np.float64)                      # :286  Float -> Double
    rho = np.ascontiguousarray(rho128, np.float64)
    finite = np.isfinite(emb32).all(axis=1)               # :591-611
    idx = np.nonzero(finite)[0]
    if idx.size == 0:
        idx = np.arange(feats.shape[0])
    train, train_rho = feats[idx], rho[idx]
    if train.shape[0] >= 2:
        initial = ahc_cluster(train, threshold, use_ref=use_ref)
    else:
        initial = np.zeros(train.shape[0], np.int32)
    vbx = vbx_refine(train_rho, psi, initial, Fa, Fb, max_iterations, epsilon)
    adjusted, detected = False, len(set(vbx.hard.tolist())) if vbx.hard.size else 0      # assignedClusterCount
    cents = None
    if (num_speakers is not None or min_speakers is not None or max_speakers is not None) and train_rho.size and initial.size:
        lo, hi = speaker_constraints(train.shape[0], num_speakers, min_speakers, max_speakers)
        if detected < lo or detected > hi:
            target = lo if detected < lo else hi
            km_labels, cents, _ = kmeans_ninit(train, target, 100, 10, 0)               # :715-721
            vbx = VBxOutput(vbx.gamma, vbx.pi, km_labels, target, vbx.elbos)
            adjusted = True                                                              # centroids used directly (:622-629)
    if cents is None:
        cents = compute_centroids(train, vbx, initial)
    if cents.shape[0] == 0:
        cents = feats.mean(axis=0, keepdims=True)         # computeFallbackCentroids :748-786
    if chunk_indices is not None and cents.shape[0] > 1 and not adjusted:
        _, scores = assign_embeddings(feats, cents, want_scores=True)
        labels = constrained_assign(scores, chunk_indices)
    else:
        labels = assign_embeddings(feats, cents)
    return ClusterResult(labels, initial, vbx, cents, idx, adjusted, detected)
