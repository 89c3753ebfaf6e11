"""mel_core.cuh's per-lane FFT / recombination / banded mel / log (the code mel512_kernel runs), emulated lane by lane on
the host (tests/emul/mel_emul.cpp) across window lengths and placements, hops and mel counts, against the oracle.  No
GPU needed: the centred and offset-0 window placements exercise both pass-1 variants (the in-window select on every slot,
and the full-middle shortcut) and the per-lane window tables for windows other than the default 400.

Bars as tests/test_gpu_config_space.py: FP64 transform within 1e-4; the float32-pair transform within
max(1e-4, 2 max |oracle(float32 FFT) - oracle|) over the same input (floor 5e-4 without pre-emphasis).
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from fluidaudio_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MEL_TOL = 1e-4
# Without pre-emphasis a frame keeps its full dynamic range and the float32 transform's noise floor shows in weak bins
# at up to ~4e-4 (512 mels, offset-0 windows), where the independent float32 FFT can happen to land closer
F32_FLOOR_NO_PREEMPH = 5e-4

WINS = [2, 64, 255, 383, 384, 449, 512]
HOPS = [2, 6, 162, 512, 1024]
N_MELS = [1, 5, 81, 257, 512]


@pytest.fixture(scope="module")
def emul(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("emul") / "libmel_emul.so")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-o", out,
                           os.path.join(ROOT, "tests", "emul", "mel_emul.cpp")])
    L = C.CDLL(out)
    f32p = np.ctypeslib.ndpointer(np.float32, flags="C_CONTIGUOUS")
    for f in (L.mel_emul, L.mel_emul_f32x2):
        f.argtypes = [f32p, C.c_longlong, C.c_float, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_int, f32p,
                      f32p, C.c_float, C.c_int, C.c_longlong, f32p]
    return L


def _check(got, ref, ref32, what, f32_floor=MEL_TOL):
    """got / ref / ref32: [frames x n_mels]."""
    d = np.abs(got.astype(np.float64) - ref)
    if ref32 is None:
        assert d.max() <= MEL_TOL, (what, float(d.max()))
    else:
        # float32 transform noise is ~0.5 ulp of a frame's largest line in every bin and lands differently in every FFT:
        # the worst element within twice the worst departure of an independent float32 FFT on the same input
        bar = max(f32_floor, 2.0 * float(np.abs(ref32.astype(np.float64) - ref).max()))
        assert d.max() <= bar, (what, float(d.max()), bar)


@pytest.mark.parametrize("win", WINS)
def test_lane_math_across_windows_hops_and_mel_counts(emul, oracle, win):
    for h, hop in enumerate(HOPS):
        for j, nm in enumerate(N_MELS):
            k = h + j + win
            frames = (17, 32, 3)[k % 3]
            gen = (synth.tone_noise_audio, synth.speech_like_audio)[k % 2]
            periodic = bool(k & 1)
            window = oracle.hann_window(win, periodic)
            fb = oracle.mel_filterbank(512, nm)
            for off in ((512 - win) // 2, 0):
                if off:    # centred window, centre padding, pre-emphasis (computeFlatTransposed)
                    n = max(1, (frames - 1) * hop + win - 512 + k % 4)
                    a = gen(n)
                    cfg = dict(n_mels=nm, hop_length=hop, win_length=win, window_periodic=periodic)
                    ref, T, _ = oracle.mel_flat_transposed(oracle.mel_config(**cfg), a, last=0.3)
                    ref32, _, _ = oracle.mel_flat_transposed(oracle.mel_config(precision=2, **cfg), a, last=0.3)
                    pad, preemph, last = 256, 0.97, 0.3
                else:      # window at offset 0, no padding, no pre-emphasis (legacy compute())
                    n = (frames - 1) * hop + win + k % 4
                    a = gen(n)
                    cfg = dict(n_mels=nm, hop_length=hop, win_length=win, window_periodic=periodic, preemph=0.0)
                    ref, T = oracle.mel_legacy(oracle.mel_config(**cfg), a)
                    ref32, _ = oracle.mel_legacy(oracle.mel_config(precision=2, **cfg), a)
                    ref, ref32 = ref.T, ref32.T
                    pad, preemph, last = 0, 0.0, 0.0
                for name, fn in (("fp64", emul.mel_emul), ("f32x2", emul.mel_emul_f32x2)):
                    out = np.zeros((T, nm), np.float32)
                    assert fn(a, a.size, np.float32(last), hop, win, off, pad, np.float32(preemph), nm, fb, window,
                              np.float32(2.0 ** -24), 0, T, out) == 0
                    _check(out, ref, ref32 if name == "f32x2" else None, (name, win, off, hop, nm, periodic),
                           MEL_TOL if preemph else F32_FLOOR_NO_PREEMPH)
