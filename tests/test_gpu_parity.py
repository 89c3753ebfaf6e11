"""GPU parity tests (run with ``-m gpu`` on the B200 box).  Every call goes through the C ABI of
libfluidaudio_b200.so (via the ctypes mirror in fluidaudio_b200/); the oracle is only the checker.

Bars (BASELINE.json north_star): cluster labels and dendrograms BIT-EXACT; log-mel and float distances within 1e-4
(tolerance spelled out as MEL_TOL below); frame counts, shapes and guards exact.
"""
import hashlib
import json
import os
import subprocess
import sys
import threading

import numpy as np
import pytest

from fluidaudio_b200 import _lib, synth
from fluidaudio_b200 import clustering as cl
from fluidaudio_b200.mel import AudioMelSpectrogram, LogFloorMode, PaddingMode, Precision

pytestmark = pytest.mark.gpu

MEL_TOL = 1e-4          # |log-mel(GPU) - log-mel(oracle)| <= 1e-4, north_star's stated tolerance
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ================================================================================================ mel
def test_mel_tables_are_bit_identical_to_the_oracle(gpu_lib, oracle):
    for nm, periodic in ((128, False), (80, False), (80, True), (23, False)):
        m = AudioMelSpectrogram(n_mels=nm, window_periodic=periodic)
        assert np.array_equal(m.get_hann_window(), oracle.hann_window(400, periodic))
        assert np.array_equal(m.get_filterbank(), oracle.mel_filterbank(512, nm))
    # reference structural tests (AudioMelSpectrogramTests.swift:57-103)
    w = AudioMelSpectrogram().get_hann_window()
    assert w.size == 400 and abs(w[0]) < 1e-6 and abs(w[-1]) < 1e-6 and abs(w[200] - 1) < 0.01
    fb = AudioMelSpectrogram().get_filterbank()
    assert fb.shape == (128, 257) and (fb >= 0).all()


@pytest.mark.parametrize("n_mels", [80, 128])
def test_mel_center_mode_lengths_and_values(gpu_lib, oracle, n_mels):
    m = AudioMelSpectrogram(n_mels=n_mels)
    cfg = oracle.mel_config(n_mels=n_mels)
    for n in (1, 2, 159, 160, 161, 399, 400, 401, 512, 4000, 5119, 5120, 16000 * 3 + 137, 16000 * 30):
        a = synth.tone_noise_audio(n, seed=n % 11)
        got, ml, nf = m.compute_flat_transposed(a)
        ref, rml, rnf = oracle.mel_flat_transposed(cfg, a)
        assert (ml, nf) == (rml, rnf) == (1 + (n + 112) // 160,) * 2
        assert got.size == nf * n_mels
        assert np.abs(got.reshape(nf, n_mels) - ref).max() <= MEL_TOL, n


def test_mel_golden_fixture(gpu_lib, golden_dir):
    g = np.load(os.path.join(golden_dir, "mel_oracle.npz"))
    a = g["audio"]
    for nm in (80, 128):
        got, ml, nf = AudioMelSpectrogram(n_mels=nm).compute_flat_transposed(a)
        assert np.abs(got.reshape(nf, nm) - g[f"center_{nm}"]).max() <= MEL_TOL
    got, ml = AudioMelSpectrogram(n_mels=128).compute(a)
    assert np.abs(got[0] - g["legacy_128"]).max() <= MEL_TOL
    m = AudioMelSpectrogram(n_mels=80, preemph=0.0, log_floor=1e-10, log_floor_mode=LogFloorMode.clamped,
                            window_periodic=True)
    got, ml, nf = m.compute_flat_transposed(a, padding_mode=PaddingMode.pre_padded)
    assert np.abs(got.reshape(nf, 80) - g["lseend_prepadded_80"]).max() <= MEL_TOL


def test_mel_all_entry_points_and_modes(gpu_lib, oracle):
    a = synth.tone_noise_audio(16000 * 5 + 77, seed=3)
    sp = synth.speech_like_audio(16000 * 8)
    for nm in (80, 128):
        m = AudioMelSpectrogram(n_mels=nm)
        cfg = oracle.mel_config(n_mels=nm)
        # computeFlat: mel-major, carries lastAudioSample into the pre-emphasis
        got, ml, nf = m.compute_flat(a, last_audio_sample=0.25)
        ref, rml, rnf = oracle.mel_flat(cfg, a, last=0.25)
        assert (ml, nf) == (rml, rnf) and np.abs(got.reshape(nm, nf) - ref).max() <= MEL_TOL
        # compute(): legacy, [1, nMels, T]
        got, ml = m.compute(a)
        ref, rml = oracle.mel_legacy(cfg, a)
        assert ml == rml and got.shape == (1, nm, ml) and np.abs(got[0] - ref).max() <= MEL_TOL
        # prePadded with and without an expected frame count (streaming callers)
        for exp in (None, 100, 600):
            got, ml, nf = m.compute_flat_transposed(a, last_audio_sample=-0.1, padding_mode=PaddingMode.pre_padded,
                                                    expected_frame_count=exp)
            ref, rml, rnf = oracle.mel_flat_transposed(cfg, a, last=-0.1, padding_mode=1, expected_frames=exp)
            assert (ml, nf) == (rml, rnf) and np.abs(got.reshape(nf, nm) - ref).max() <= MEL_TOL
        got, ml, nf = m.compute_flat_transposed(sp)
        ref, _, _ = oracle.mel_flat_transposed(cfg, sp)
        assert np.abs(got.reshape(nf, nm) - ref).max() <= MEL_TOL
    # padTo: padded rows are zero (AudioMelSpectrogram.swift:354,394)
    m = AudioMelSpectrogram(n_mels=80, pad_to=16)
    got, ml, nf = m.compute_flat_transposed(a[:4000])
    assert (ml, nf) == (26, 32) and np.all(got.reshape(32, 80)[26:] == 0)
    got, ml, nf = m.compute_flat(a[:4000])
    assert (ml, nf) == (26, 32) and np.all(got.reshape(80, 32)[:, 26:] == 0)
    ref, _, _ = oracle.mel_flat(oracle.mel_config(n_mels=80, pad_to=16), a[:4000])
    assert np.abs(got.reshape(80, 32) - ref).max() <= MEL_TOL
    # LS-EEND style configuration (LSEENDPreprocessor.swift:70-81) with the nFFT the reference derives from the window,
    # nFFT = nextPow2(winLength) (LSEENDTypes.swift:55-57): 200 -> 256 (8 kHz model), 400 -> 512 (16 kHz model)
    for win, hop, nfft in ((200, 80, 256), (400, 160, 512)):
        m = AudioMelSpectrogram(n_mels=23, n_fft=nfft, hop_length=hop, win_length=win, preemph=0.0, log_floor=1e-10,
                                log_floor_mode=LogFloorMode.clamped, window_periodic=True)
        cfg = oracle.mel_config(n_mels=23, n_fft=nfft, hop_length=hop, win_length=win, preemph=0.0, log_floor=1e-10,
                                log_floor_mode=1, window_periodic=True)
        got, ml, nf = m.compute_flat_transposed(sp[:40000], padding_mode=PaddingMode.pre_padded)
        ref, rml, rnf = oracle.mel_flat_transposed(cfg, sp[:40000], padding_mode=1)
        assert (ml, nf) == (rml, rnf) and np.abs(got.reshape(nf, 23) - ref).max() <= MEL_TOL


def test_mel_any_power_of_two_nfft_and_odd_hop(gpu_lib, oracle):
    """AudioMelSpectrogram is parametric (AudioMelSpectrogram.swift:59-70): nFFT 256 / 1024 / 2048, odd hops, windows
    shorter than nFFT, every entry point and both layouts — the any-nFFT kernel against the oracle at the same bar."""
    a = synth.tone_noise_audio(16000 * 3 + 41, seed=5)
    sp = synth.speech_like_audio(16000 * 3)
    cases = [dict(n_fft=256, win_length=200, hop_length=80, n_mels=23), dict(n_fft=1024, win_length=800, hop_length=320, n_mels=80),
             dict(n_fft=512, win_length=400, hop_length=161, n_mels=80), dict(n_fft=2048, win_length=1200, hop_length=441, n_mels=128),
             dict(n_fft=64, win_length=64, hop_length=17, n_mels=10), dict(n_fft=1024, win_length=1024, hop_length=256, n_mels=64,
                                                                      preemph=0.0, window_periodic=True)]
    for kw in cases:
        m = AudioMelSpectrogram(**kw)
        okw = dict(kw)
        if "window_periodic" in okw:
            okw["window_periodic"] = 1
        cfg = oracle.mel_config(**okw)
        nm, bins = kw["n_mels"], kw["n_fft"] // 2 + 1
        assert np.array_equal(m.get_filterbank(), oracle.mel_filterbank(kw["n_fft"], nm)) and m.get_filterbank().shape == (nm, bins)
        for sig in (a, sp, a[:kw["n_fft"] // 2 + 3]):
            got, ml, nf = m.compute_flat_transposed(sig, last_audio_sample=0.2)
            ref, rml, rnf = oracle.mel_flat_transposed(cfg, sig, last=0.2)
            assert (ml, nf) == (rml, rnf) and np.abs(got.reshape(nf, nm) - ref).max() <= MEL_TOL, kw
            got, ml, nf = m.compute_flat(sig)
            ref, rml, rnf = oracle.mel_flat(cfg, sig)
            assert (ml, nf) == (rml, rnf) and np.abs(got.reshape(nm, nf) - ref).max() <= MEL_TOL, kw
        got, ml, nf = m.compute_flat_transposed(a, padding_mode=PaddingMode.pre_padded)
        ref, rml, rnf = oracle.mel_flat_transposed(cfg, a, padding_mode=1)
        assert (ml, nf) == (rml, rnf) and np.abs(got.reshape(nf, nm) - ref).max() <= MEL_TOL, kw
        got, ml = m.compute(a)
        ref, rml = oracle.mel_legacy(cfg, a)
        assert ml == rml and np.abs(got[0] - ref).max() <= MEL_TOL, kw
    # batch entry point on the generic path == one by one
    m = AudioMelSpectrogram(n_fft=256, win_length=200, hop_length=80, n_mels=23)
    clips = [a[:5000], sp[:12345], a[:90]]
    out, offs, ml, nf = m.compute_batch(clips)
    for i, c in enumerate(clips):
        single, _, _ = m.compute_flat_transposed(c)
        assert np.array_equal(single, out[offs[i]:offs[i + 1]])
    for bad in (dict(n_fft=400), dict(n_fft=8192), dict(n_fft=256, win_length=400)):
        with pytest.raises(_lib.FluidAudioError) as e:
            AudioMelSpectrogram(**bad)
        assert e.value.status == 8


def test_mel_guards_silence_and_unsupported(gpu_lib):
    m = AudioMelSpectrogram(n_mels=128)
    out, ml, nf = m.compute_flat_transposed(np.zeros(0, np.float32))
    assert (ml, nf) == (0, 1) and out.size == 128 and np.all(out == 0)           # :349-351
    # legacy frame count 1 + (n - 400) / 160 uses Swift's truncating division: 300 samples still give one
    # (partially filled) frame, 200 samples give none
    assert m.compute(np.zeros(300, np.float32))[1] == 1
    assert m.compute(np.zeros(200, np.float32))[1] == 0
    mel, ml = m.compute(np.zeros(16000, np.float32))                            # AudioMelSpectrogramTests.swift:32-45,107-122
    assert ml == 98 and mel.shape == (1, 128, 98) and (mel < 0).all()
    floor = np.log(np.float32(2.0 ** -24))
    got, ml, nf = m.compute_flat_transposed(np.zeros(8000, np.float32))
    assert np.abs(got - floor).max() <= 4e-6                                    # silence is log(floor) (device log: 2 ulp)
    assert m.compute(np.full(800, 0.1, np.float32))[1] > 0                      # :24-30
    for n, frames in ((2560, 17), (20480, 129)):                                # EouChunkSizeFrameCountTests.swift
        assert m.compute_flat(np.full(n, 0.1, np.float32))[1] == frames
    with pytest.raises(_lib.FluidAudioError) as e:
        AudioMelSpectrogram(n_fft=400)
    assert e.value.status == 8


def test_mel_batch_and_device_paths(gpu_lib, oracle):
    m = AudioMelSpectrogram(n_mels=80)
    cfg = oracle.mel_config(n_mels=80)
    lens = [480000, 1000, 33333, 7, 480000, 161, 250001]
    clips = [synth.tone_noise_audio(n, seed=i) for i, n in enumerate(lens)]
    last = np.linspace(-0.2, 0.2, len(lens)).astype(np.float32)
    out, offs, ml, nf = m.compute_batch(clips, last_samples=last)
    for i, c in enumerate(clips):
        ref, rml, rnf = oracle.mel_flat_transposed(cfg, c, last=float(last[i]))
        assert (ml[i], nf[i]) == (rml, rnf)
        assert np.abs(out[offs[i]:offs[i + 1]].reshape(-1, 80) - ref).max() <= MEL_TOL
        single, _, _ = m.compute_flat_transposed(c, last_audio_sample=float(last[i]))
        assert np.array_equal(single, out[offs[i]:offs[i + 1]])                  # batch == one-by-one, bitwise
    # clips that start at multiples of four floats in the caller's buffer keep that layout on the device and travel one
    # transfer per group (BASELINE configs[3]: 512 x 480 000): lengths that are not multiples of four sit in aligned slots
    # with gaps (filled with a sentinel the kernel must never read), plus an empty clip and 40 clips -> several per group
    lens2 = [480000, 1001, 0, 33333, 6, 4000] + [16000 + 4 * i for i in range(34)]
    clips2 = [synth.tone_noise_audio(n, seed=50 + i) for i, n in enumerate(lens2)]
    offs2 = np.zeros(len(lens2) + 1, np.int64)
    starts = []
    pos = 0
    for n in lens2:
        starts.append(pos)
        pos += -(-n // 4) * 4 + (8 if n % 8 == 1 else 0)
    packed = np.full(pos + 4, 1e30, np.float32)
    for st, c in zip(starts, clips2):
        packed[st:st + c.size] = c
    # the C entry point takes offsets[i], offsets[i+1] as the clip's bounds: pass exact ends through a second call shape
    ends = [st + c.size for st, c in zip(starts, clips2)]
    for i, (st, en) in enumerate(zip(starts, ends)):
        single, ml1, nf1 = m.compute_flat_transposed(clips2[i]) if clips2[i].size else (None, 0, 1)
        if clips2[i].size:
            # one-clip "batch" at an aligned start inside the sentinel-padded buffer
            o1, oo1, mlb, nfb = m.compute_batch(None, packed_audio=packed[st:], offsets=np.array([0, en - st], np.int64))
            assert (mlb[0], nfb[0]) == (ml1, nf1) and np.array_equal(o1[oo1[0]:oo1[1]], single)
    aligned = [c for c in clips2 if c.size % 4 == 0]                              # contiguous AND aligned: the grouped path
    outb, offb, mlb, nfb = m.compute_batch(aligned)
    for i, c in enumerate(aligned):
        if c.size == 0:
            continue
        single, ml1, nf1 = m.compute_flat_transposed(c)
        assert (mlb[i], nfb[i]) == (ml1, nf1) and np.array_equal(outb[offb[i]:offb[i + 1]], single), i
    # device-resident entry point == host entry point, bitwise; unaligned device pointers take the non-TMA path
    a = clips[0]
    T = m.frame_count(a.size)
    host, _, _ = m.compute_flat_transposed(a)
    d_a = _lib.DeviceBuffer(a.nbytes + 64)
    d_o = _lib.DeviceBuffer(T * 80 * 4)
    d_a.upload(a)
    assert m.compute_device(d_a, a.size, d_o) == (T, T)
    _lib.synchronize()
    assert np.array_equal(d_o.download((T * 80,), np.float32), host)
    shifted = np.concatenate([np.zeros(1, np.float32), a])
    d_a.upload(shifted)

    class Off:                                                                  # view of the buffer at +4 bytes
        ptr = d_a.ptr.value + 4
    ml2, nf2 = m.compute_device(Off, a.size, d_o)
    _lib.synchronize()
    assert np.array_equal(d_o.download((T * 80,), np.float32), host)


def test_mel_pipeline_knobs_do_not_change_results(gpu_lib):
    """fa_mel_set_pipeline_chunks / fa_mel_set_zero_copy_output only move data differently: every depth, the kernel storing
    straight into the caller's pinned buffer or staging + D2H, float32 and int16 PCM entry points — bit-identical rows."""
    n = 16000 * 150
    a = synth.tone_noise_audio(n)
    pin_in = _lib.PinnedArray(n, np.float32); pin_in.array[:] = a
    pin_16 = _lib.PinnedArray(n, np.int16); pin_16.array[:] = np.round(a * 32767).astype(np.int16)
    for prec in (Precision.f64, Precision.f32):
        m = AudioMelSpectrogram(n_mels=80, precision=prec)
        T = m.frame_count(n)
        pin_out = _lib.PinnedArray(T * 80, np.float32)
        ref, _, _ = m.compute_flat_transposed(a)                     # pageable buffers, default depth
        ref16, _, _, _ = m.compute_from_pcm(pin_16.array.copy(), 16000.0)
        for zc in (0, 1):
            _lib.check(m._L.fa_mel_set_zero_copy_output(m._h, zc), "zero copy")
            for chunks in (1, 2, 7, 24, 200):
                _lib.check(m._L.fa_mel_set_pipeline_chunks(m._h, chunks), "chunks")
                pin_out.array[:] = -1.0
                got, ml, nf = m.compute_flat_transposed(pin_in.array, out=pin_out.array)
                assert np.array_equal(got, ref), (prec, zc, chunks)
                pin_out.array[:] = -1.0
                got, ml, nf, rs = m.compute_from_pcm(pin_16.array, 16000.0, out=pin_out.array)
                assert rs == n and np.array_equal(got, ref16), (prec, zc, chunks)
    with pytest.raises(_lib.FluidAudioError):
        _lib.check(m._L.fa_mel_set_pipeline_chunks(m._h, 0), "chunks")


def test_mel_one_hour_properties(gpu_lib, oracle):
    """BASELINE config 2 at full size: 1 h of 16 kHz audio, 80 mels."""
    n = 57_600_000
    a = synth.tone_noise_audio(n)
    m = AudioMelSpectrogram(n_mels=80)
    T = m.frame_count(n)
    assert T == 360001
    host, ml, nf = m.compute_flat_transposed(a)                                 # chunked H2D / kernel / D2H pipeline
    host = host.reshape(T, 80)
    d_a = _lib.DeviceBuffer(n * 4 + 64)
    d_o = _lib.DeviceBuffer(T * 80 * 4)
    d_a.upload(a)
    m.compute_device(d_a, n, d_o)                                               # one launch over all frames
    _lib.synchronize()
    assert np.array_equal(d_o.download((T, 80), np.float32), host)              # chunking is invisible, bitwise
    assert np.isfinite(host).all()
    # a frame depends only on its own 400 samples: excerpts starting on a hop boundary reproduce interior frames
    for start_frame in (0, 1000, 123456, 359000):
        s0 = start_frame * 160
        ex = a[s0:s0 + 16000 * 5]
        sub, sml, _ = m.compute_flat_transposed(ex, last_audio_sample=float(a[s0 - 1]) if s0 else 0.0)
        sub = sub.reshape(sml, 80)
        assert np.array_equal(sub[2:sml - 3], host[start_frame + 2:start_frame + sml - 3])
    # against the oracle: the first minute and a window in the middle
    cfg = oracle.mel_config(n_mels=80)
    ref, rml, _ = oracle.mel_flat_transposed(cfg, a[:960000])
    assert np.abs(host[:rml - 3] - ref[:rml - 3]).max() <= MEL_TOL
    s0 = 200000 * 160
    ref, rml, _ = oracle.mel_flat_transposed(cfg, a[s0:s0 + 960000], last=float(a[s0 - 1]))
    assert np.abs(host[200000 + 2:200000 + rml - 3] - ref[2:rml - 3]).max() <= MEL_TOL


def test_mel_float32_transform_option(gpu_lib, oracle):
    """FA_MEL_PRECISION_F32: the transform in float32 like the reference's vDSP_DFT (two frames per warp, packed
    FFMA2).  Same entry points, shapes and guards; values within the SAME 1e-4 bar on BASELINE's signal — checked over
    the WHOLE hour against the FP64 path (itself within 5e-6 of the oracle) and directly against the oracle on windows."""
    n = 57_600_000
    a = synth.tone_noise_audio(n)
    m64 = AudioMelSpectrogram(n_mels=80)
    m32 = AudioMelSpectrogram(n_mels=80, precision=Precision.f32)
    assert m32._L.fa_mel_get_precision(m32._h) == 1 and m64._L.fa_mel_get_precision(m64._h) == 0
    h64, ml, nf = m64.compute_flat_transposed(a)
    h32, ml2, nf2 = m32.compute_flat_transposed(a)
    assert (ml, nf) == (ml2, nf2) == (360001, 360001)
    d = np.abs(h32 - h64)
    assert np.isfinite(h32).all() and d.max() <= MEL_TOL, d.max()
    cfg = oracle.mel_config(n_mels=80)
    h32 = h32.reshape(ml, 80)
    ref, rml, _ = oracle.mel_flat_transposed(cfg, a[:960000])
    assert np.abs(h32[:rml - 3] - ref[:rml - 3]).max() <= MEL_TOL
    # every mode / layout / odd length, 128 mels, the harder fixture; frames are independent of their pair partner
    sp = synth.speech_like_audio(16000 * 8)
    m = AudioMelSpectrogram(n_mels=128, precision=Precision.f32)
    cfg = oracle.mel_config(n_mels=128)
    for sig in (sp, synth.tone_noise_audio(16000 * 5 + 77, seed=3), synth.tone_noise_audio(161), synth.tone_noise_audio(7)):
        got, ml, nf = m.compute_flat_transposed(sig)
        ref, rml, rnf = oracle.mel_flat_transposed(cfg, sig)
        assert (ml, nf) == (rml, rnf) and np.abs(got.reshape(nf, 128) - ref).max() <= MEL_TOL
        got, ml, nf = m.compute_flat(sig, last_audio_sample=0.25)
        ref, rml, rnf = oracle.mel_flat(cfg, sig, last=0.25)
        assert (ml, nf) == (rml, rnf) and np.abs(got.reshape(128, nf) - ref).max() <= MEL_TOL
    # legacy compute(): NO pre-emphasis, so the 60 dB fixture keeps its full dynamic range in one frame and the float32
    # noise floor of ANY float32 FFT (0.5 ulp of the strongest harmonic in every bin) shows: 1.4e-4 measured.  This is why
    # the FP64 transform is the library default; the float32 option is held to 3e-4 here and to 1e-4 everywhere else.
    got, ml = m.compute(sp)
    ref, rml = oracle.mel_legacy(cfg, sp)
    assert ml == rml and np.abs(got[0] - ref).max() <= 3e-4
    got, ml, nf = m.compute_flat_transposed(sp, last_audio_sample=-0.1, padding_mode=PaddingMode.pre_padded, expected_frame_count=333)
    ref, rml, rnf = oracle.mel_flat_transposed(cfg, sp, last=-0.1, padding_mode=1, expected_frames=333)
    assert (ml, nf) == (rml, rnf) and np.abs(got.reshape(nf, 128) - ref).max() <= MEL_TOL
    ex = sp[160 * 100:160 * 100 + 16000]
    sub, sml, _ = m.compute_flat_transposed(ex, last_audio_sample=float(sp[160 * 100 - 1]))
    full, fml, _ = m.compute_flat_transposed(sp)
    assert np.array_equal(sub.reshape(sml, 128)[2:sml - 3], full.reshape(fml, 128)[102:100 + sml - 3])
    with pytest.raises(_lib.FluidAudioError):
        m.set_precision(7)


def test_swift_goldens_when_present(gpu_lib, golden_dir):
    """Apple's own numbers (swift/Tools/DumpGoldens.swift run on a Mac, packed by tests/golden/swift_fixtures.py) against the
    CUDA path.  Absent in this repository (no Swift toolchain): the test then skips and mel / VBx VALUES stay "parity
    unpinned" against the reference binary, as DESIGN.md states."""
    mel_path, vbx_path = os.path.join(golden_dir, "swift_mel.npz"), os.path.join(golden_dir, "swift_vbx.npz")
    if not (os.path.exists(mel_path) or os.path.exists(vbx_path)):
        pytest.skip("parity unpinned: no Swift-run goldens (tests/golden/swift_*.npz)")
    if os.path.exists(mel_path):
        g = np.load(mel_path)
        for prec in (Precision.f64, Precision.f32):
            for name in ("tone_noise", "speech_like"):
                for nm in (80, 128):
                    m = AudioMelSpectrogram(n_mels=nm, precision=prec)
                    got, ml, nf = m.compute_flat_transposed(g[f"audio_{name}"])
                    assert [ml, nf] == g[f"{name}_{nm}_center_shape"].tolist()
                    assert np.abs(got - g[f"{name}_{nm}_center"]).max() <= 2e-4
    if os.path.exists(vbx_path):
        g = np.load(vbx_path)
        out = cl.VBxClustering(psi=g["psi"]).refine(g["rho"], g["initial"])
        assert np.array_equal(np.asarray(out.hard_clusters, np.int32).reshape(-1), g["hard"].reshape(-1))
        assert np.abs(out.gamma - g["gamma"]).max() <= 1e-6


# ================================================================================================ AudioConverter (R1)
def _sine_pcm(rate, channels, seconds, seed=0):
    """AudioConverterTests.swift createAudioBuffer: a 440 Hz sine of amplitude 0.5 per channel (here each channel gets its
    own frequency and a little noise so that a wrong mixdown or channel order cannot hide)."""
    rng = np.random.default_rng(seed)
    t = np.arange(int(rate * seconds)) / rate
    return np.stack([(0.5 * np.sin(2 * np.pi * (440.0 + 110.0 * c) * t) + 0.01 * rng.standard_normal(t.size)).astype(np.float32)
                     for c in range(channels)])


def test_audio_converter_reference_tests_and_filter_spec(gpu_lib, oracle):
    from fluidaudio_b200.audio_converter import AudioConverter
    conv = AudioConverter()
    # testConvertAlreadyCorrectFormat / resample(_:from:) identity (:66-68): same samples, bit for bit
    x = _sine_pcm(16000, 1, 1.0)[0]
    assert np.array_equal(conv.resample(x, 16000), x) and conv.resample(np.zeros(0, np.float32), 48000).size == 0
    assert np.array_equal(conv.resample_buffer(x[None], 16000), x)
    # lengths: 44.1k stereo 1 s, 48k mono 0.5 s, 8k mono 2 s within 1 % (AudioConverterTests.swift:129-176); short buffer
    for rate, ch, dur, expect in ((44100, 2, 1.0, 16000), (48000, 1, 0.5, 8000), (8000, 1, 2.0, 32000), (44100, 1, 0.01, 160)):
        y = conv.resample_buffer(_sine_pcm(rate, ch, dur), rate)
        assert y.size > 0 and abs(y.size - expect) <= 0.01 * expect + 1 and np.abs(y).max() <= 0.6
        assert y.size == oracle.resample_output_count(int(rate * dur), rate, 16000) == conv.output_count(int(rate * dur), rate)
    # testConvertStereoToMono: same rate, 1000 frames -> 1000 frames, mean of the channels
    st = _sine_pcm(16000, 2, 1000 / 16000)
    assert np.array_equal(conv.resample_buffer(st, 16000), oracle.mixdown(st))
    # values against the float64 evaluation of the documented filter (float32 taps and sums: <= 3e-6 of full scale)
    for rate in (8000, 11025, 22050, 32000, 44100, 48000, 96000, 16001):
        m = _sine_pcm(rate, 1, 0.35, seed=rate)[0]
        got = conv.resample(m, rate)
        ref = oracle.sinc_resample(m, rate, 16000)
        assert got.shape == ref.shape and np.abs(got - ref).max() <= (2e-5 if rate == 16001 else 3e-6), rate
    # stereo, int16, interleaved and planar: mixdown + widening happen on the device
    st = _sine_pcm(44100, 2, 0.4, seed=5)
    i16 = np.round(st * 32767).astype(np.int16)
    ref = oracle.sinc_resample(oracle.mixdown(i16), 44100, 16000)
    assert np.abs(conv.resample_buffer(i16, 44100) - ref).max() <= 3e-6
    assert np.array_equal(conv.resample_buffer(np.ascontiguousarray(i16.T), 44100, interleaved=True), conv.resample_buffer(i16, 44100))
    assert np.abs(conv.resample_buffer(st, 44100) - oracle.sinc_resample(oracle.mixdown(st), 44100, 16000)).max() <= 3e-6
    # > 2 channels: AudioConverter.linearResample, bit for bit (planar float32 as floatChannelData; interleaved too)
    for ch, rate in ((3, 44100), (4, 48000), (6, 8000), (5, 16000)):
        p = _sine_pcm(rate, ch, 0.2, seed=ch)
        ref = oracle.linear_resample(p, rate, 16000)
        assert np.array_equal(conv.resample_buffer(p, rate), ref)
        assert np.array_equal(conv.resample_buffer(np.ascontiguousarray(p.T), rate, interleaved=True), ref)
    # a tone above the new Nyquist is gone, one below it keeps its amplitude (what "Mastering quality" must deliver)
    t = np.arange(48000) / 48000.0
    for f0, lo, hi in ((1000.0, 0.4999, 0.5001), (10000.0, 0.0, 2e-6)):
        y = conv.resample((0.5 * np.sin(2 * np.pi * f0 * t)).astype(np.float32), 48000)[2000:-2000]
        amp = np.sqrt(2.0 * np.mean(y.astype(np.float64) ** 2))
        assert lo <= amp <= hi, (f0, amp)
    # guards
    with pytest.raises(_lib.FluidAudioError):
        conv.resample_buffer(np.zeros((65, 10), np.float32), 48000)


def test_audio_to_mel_fused_pipeline(gpu_lib, oracle):
    """fa_audio_to_mel == fa_mel_compute(fa_audio_resample(pcm)) bit for bit (the chunked PCM pipeline is invisible),
    for float32 / int16, mono / stereo / 4 channels, every rate; 16 kHz mono float32 is the plain mel path."""
    from fluidaudio_b200.audio_converter import AudioConverter
    conv = AudioConverter()
    m = AudioMelSpectrogram(n_mels=80)
    cases = [(48000, 1, np.float32, 3.0), (44100, 2, np.int16, 2.5), (8000, 1, np.int16, 4.0), (48000, 4, np.float32, 1.0),
             (16000, 1, np.int16, 2.0), (16000, 2, np.float32, 1.5), (16000, 1, np.float32, 1.0), (22050, 1, np.float32, 20.0)]
    for rate, ch, dt, dur in cases:
        p = _sine_pcm(rate, ch, dur, seed=rate + ch)
        if dt == np.int16:
            p = np.round(p * 32767).astype(np.int16)
        inter = np.ascontiguousarray(p.T)
        mono = conv.resample_buffer(p, rate)
        ref, rml, rnf = m.compute_flat_transposed(mono, last_audio_sample=0.1)
        got, ml, nf, rs = m.compute_from_pcm(inter, rate, interleaved=True, last_audio_sample=0.1)
        assert (ml, nf, rs) == (rml, rnf, mono.size) and np.array_equal(got, ref), (rate, ch)
        got2, _, _, _ = m.compute_from_pcm(p, rate, last_audio_sample=0.1, time_major=False)
        assert np.array_equal(got2.reshape(80, nf).T, ref.reshape(nf, 80))
    # the whole chain against the oracle: oracle filter (float64) -> oracle mel, within the mel bar
    x = synth.tone_noise_audio(48000 * 4)[: 48000 * 4]
    up = oracle.sinc_resample(x, 16000, 48000)          # a 48 kHz rendition of the fixture
    got, ml, nf, rs = m.compute_from_pcm(up, 48000)
    ref, rml, _ = oracle.mel_flat_transposed(oracle.mel_config(n_mels=80), oracle.sinc_resample(up, 48000, 16000))
    assert ml == rml and np.abs(got.reshape(nf, 80) - ref).max() <= 2e-3   # float32 filter sums ahead of a log
    with pytest.raises(_lib.FluidAudioError):
        AudioMelSpectrogram(n_mels=80, sample_rate=8000).compute_from_pcm(np.zeros(100, np.float32), 16000, algorithm=9)


# ================================================================================================ AHC
def _ref_linkage(oracle, x):
    return oracle.centroid_linkage(x, use_ref=True)


def test_linkage_reproduces_reference_goldens_bit_exact(gpu_lib, golden_dir):
    g = np.load(os.path.join(golden_dir, "ahc_reference.npz"))
    for name in sorted({k.rsplit("__", 1)[0] for k in g.files}):
        st, z = cl.centroid_linkage(g[name + "__x"])
        assert st == 0 and np.array_equal(z, g[name + "__z"]), name


def test_linkage_bit_exact_on_fresh_inputs_and_status_codes(gpu_lib, oracle):
    rng = np.random.default_rng(99)
    for n, d in ((2, 1), (3, 2), (33, 5), (129, 256), (1000, 64), (2049, 256), (777, 300), (64, 1023)):
        x = rng.standard_normal((n, d))
        st, z = cl.centroid_linkage(x)
        st2, z2 = _ref_linkage(oracle, x)
        assert st == st2 == 0 and np.array_equal(z, z2), (n, d)
    x = np.round(rng.standard_normal((400, 4)), 1)                               # masses of exactly tied distances
    assert np.array_equal(cl.centroid_linkage(x)[1], _ref_linkage(oracle, x)[1])
    x = np.repeat(rng.standard_normal((40, 6)), 5, axis=0)[rng.permutation(200)]  # duplicates: zero distances
    assert np.array_equal(cl.centroid_linkage(x)[1], _ref_linkage(oracle, x)[1])
    bad = rng.standard_normal((50, 8)); bad[17, 3] = np.nan
    assert cl.centroid_linkage(bad)[0] == 5                                      # nan_error -> RUNTIME_ERROR
    inf = rng.standard_normal((20, 4)); inf[3, 0] = np.inf; inf[9, 0] = np.inf   # inf - inf = NaN
    assert cl.centroid_linkage(inf)[0] == _ref_linkage(oracle, inf)[0] == 5
    one_inf = rng.standard_normal((20, 4)); one_inf[3, 0] = np.inf               # infinite but never NaN
    st, z = cl.centroid_linkage(one_inf)
    st2, z2 = _ref_linkage(oracle, one_inf)
    assert st == st2 and (st != 0 or np.array_equal(z, z2))
    L = gpu_lib
    zbuf = np.zeros(8)
    assert L.fastcluster_compute_centroid_linkage(np.ones((3, 2)).ctypes.data, 3, 2, zbuf.ctypes.data, 7) == 3


def test_linkage_fallback_placements_are_bit_exact(gpu_lib, oracle):
    """Master state in global memory / node vectors streamed from L2 (the large-N code paths) at small N."""
    code = (
        "import sys, numpy as np; sys.path.insert(0, %r);"
        "from fluidaudio_b200 import clustering as cl; from oracle import oracle as O;"
        "rng = np.random.default_rng(5);"
        "ok = True\n"
        "for n, d in ((3, 2), (300, 16), (1500, 256)):\n"
        "    x = rng.standard_normal((n, d)); st, z = cl.centroid_linkage(x); st2, z2 = O.centroid_linkage(x)\n"
        "    ok = ok and st == 0 and np.array_equal(z, z2)\n"
        "print('FALLBACK_OK' if ok else 'FALLBACK_BAD')" % ROOT)
    for env in ({"FA_AHC_FORCE_GLOBAL_MASTER": "1"}, {"FA_AHC_FORCE_STREAMED": "1"},
                {"FA_AHC_FORCE_GLOBAL_MASTER": "1", "FA_AHC_FORCE_STREAMED": "1"}):
        out = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, **env), capture_output=True, text=True,
                             timeout=600)
        assert "FALLBACK_OK" in out.stdout, (env, out.stdout[-500:], out.stderr[-1500:])


def test_linkage_float32_filter_is_bit_exact(gpu_lib, golden_dir, oracle):
    """The float32 GEMM-form filter of the initial nearest-neighbour pass (ahc_filter_*_kernel: rigorous error bound,
    exact chains only for candidates) forced on at every size (FA_AHC_FILTER_MIN_N=2): the reference's goldens — exact
    ties on a lattice, duplicates, a line — and fresh inputs incl. zero vectors, huge and non-finite values (which must
    fall back to the exact pass and keep the reference's status codes) stay bit-identical."""
    code = (
        "import sys, os, numpy as np; sys.path.insert(0, %r);"
        "from fluidaudio_b200 import clustering as cl; from oracle import oracle as O;"
        "g = np.load(os.path.join(%r, 'ahc_reference.npz')); ok = True\n"
        "for k in [k[:-3] for k in g.files if k.endswith('__x')]:\n"
        "    st, z = cl.centroid_linkage(g[k + '__x']); ok = ok and st == 0 and np.array_equal(z, g[k + '__z'])\n"
        "rng = np.random.default_rng(9)\n"
        "cases = [rng.standard_normal((700, 64)), np.repeat(rng.standard_normal((40, 8)), 30, axis=0), rng.standard_normal((513, 256)) * 1e-9,"
        " np.concatenate([np.zeros((5, 16)), rng.standard_normal((300, 16))]), rng.standard_normal((200, 16)) * 1e30]\n"
        "from fluidaudio_b200 import synth\n"
        "e, _ = synth.speaker_embeddings(3000, 256, 4, seed=2); cases.append(O.l2_normalize_rows(e.astype(np.float64)))\n"
        "for x in cases:\n"
        "    st, z = cl.centroid_linkage(x); st2, z2 = O.centroid_linkage(x, use_ref=True); ok = ok and st == st2 and np.array_equal(z, z2)\n"
        "bad = rng.standard_normal((100, 8)); bad[50, 3] = np.nan\n"
        "ok = ok and cl.centroid_linkage(bad)[0] == O.centroid_linkage(bad, use_ref=True)[0] == 5\n"
        "print('FILTER_OK' if ok else 'FILTER_BAD')" % (ROOT, golden_dir))
    for env in ({"FA_AHC_FILTER_MIN_N": "2"}, {"FA_AHC_FILTER_MIN_N": "0"}):
        out = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, **env), capture_output=True, text=True, timeout=900)
        assert "FILTER_OK" in out.stdout, (env, out.stdout[-500:], out.stderr[-1500:])


def test_linkage_is_reentrant(gpu_lib, oracle):
    rng = np.random.default_rng(4)
    xs = [rng.standard_normal((400 + 50 * i, 32)) for i in range(6)]
    want = [oracle.centroid_linkage(x)[1] for x in xs]
    got = [None] * len(xs)

    def run(i):
        got[i] = cl.centroid_linkage(xs[i])

    threads = [threading.Thread(target=run, args=(i,)) for i in range(len(xs))]
    [t.start() for t in threads]
    [t.join() for t in threads]
    for i in range(len(xs)):
        assert got[i][0] == 0 and np.array_equal(got[i][1], want[i])


def test_ahc_cluster_reference_unit_tests(gpu_lib, oracle):
    """AHCClusteringTests.swift through the GPU path."""
    ahc = cl.AHCClustering()
    assert ahc.cluster([], 0.7).size == 0
    assert ahc.cluster([[1.0, 0.0, 0.0]], 0.7).tolist() == [0]
    assert len(set(ahc.cluster([[1.0, 2.0, 3.0]] * 5, 0.7).tolist())) == 1
    g1 = [[1.0, 0, 0], [0.9, 0.1, 0], [0.95, 0.05, 0]]
    g2 = [[0, 1.0, 0], [0, 0.9, 0.1], [0, 0.95, 0.05]]
    r = ahc.cluster(g1 + g2, 0.8)
    assert len(set(r[:3].tolist())) == 1 and len(set(r[3:].tolist())) == 1 and r[0] != r[3]
    four = [[1.0, 0, 0], [0.9, 0.1, 0], [0, 1.0, 0], [0, 0.9, 0.1]]
    assert len(set(ahc.cluster(four, 0.5).tolist())) == 2 and len(set(ahc.cluster(four, 1.5).tolist())) == 1
    eye = np.eye(3)
    ids = sorted(set(ahc.cluster(eye, 0.5).tolist()))
    assert ids == list(range(len(ids)))
    assert len(set(ahc.cluster(eye, 2.0).tolist())) == 1 and len(set(ahc.cluster(eye, 0.0).tolist())) == 3
    assert ahc.cluster(np.zeros((3, 0)), 0.7).tolist() == [0, 0, 0]
    nan_rows = np.array([[1.0, 0.0], [np.nan, 1.0], [0.0, 1.0]])
    assert ahc.cluster(nan_rows, 0.7).tolist() == [0, 1, 2]                      # FFI failure -> identity (:52-55)
    rng = np.random.default_rng(8)
    for n in (5, 50, 700):
        x = rng.standard_normal((n, 16)) + 3 * rng.integers(0, 3, (n, 1))
        for thr in (0.0, 0.4, 0.9, 1.3, 2.0, 7.0, -2.0, float("nan")):
            assert np.array_equal(ahc.cluster(x, thr), oracle.ahc_cluster(x, thr))
    assert np.array_equal(cl.l2_normalize_rows(x), oracle.l2_normalize_rows(x))  # same operation order: bitwise


def test_baseline_size_problems_match_reference_hashes(gpu_lib, golden_dir, oracle):
    """C5 (5 000 x 256) and C3 (10 000 x 256): dendrogram bytes and labels hashed against the reference run."""
    meta = json.load(open(os.path.join(golden_dir, "ahc_large.json")))
    for name, m in meta.items():
        emb, _ = synth.speaker_embeddings(m["n"], 256, m["speakers"], weights=m["weights"], seed=m["seed"])
        x = oracle.l2_normalize_rows(emb.astype(np.float64))
        st, z = cl.centroid_linkage(x)
        assert st == 0
        assert hashlib.sha256(z.tobytes()).hexdigest() == m["z_sha256"], name
        labels = cl.dendrogram_cut(z, m["n"], 0.6)
        assert hashlib.sha256(labels.tobytes()).hexdigest() == m["labels_sha256"]
        assert np.array_equal(cl.AHCClustering().cluster(emb.astype(np.float64), 0.6), labels)
        rho, psi = synth.synthetic_plda(emb)
        res = cl.OfflineClusterer(psi=psi).cluster(emb, rho)
        assert hashlib.sha256(res.labels.tobytes()).hexdigest() == m["final_labels_sha256"], name
        assert res.info["centroid_count"] == m["final_centroids"]
        assert res.info["vbx_iterations"] == m["vbx_iterations"]
        # size-independent properties: sizes telescope to N, every node id appears exactly once as a child
        assert z[-1, 3] == m["n"]
        kids = np.concatenate([z[:, 0], z[:, 1]]).astype(np.int64)
        assert np.array_equal(np.sort(kids), np.arange(2 * m["n"] - 2))


# ================================================================================================ VBx / pipeline
def test_vbx_centroids_assignment_against_oracle(gpu_lib, oracle):
    for n, k, seed in ((300, 3, 1), (1500, 6, 2), (4000, 8, 3)):
        emb, _ = synth.speaker_embeddings(n, 256, k, seed=seed)
        rho, psi = synth.synthetic_plda(emb)
        init = oracle.ahc_cluster(emb.astype(np.float64), 0.6)
        o = oracle.vbx_refine(rho, psi, init)
        v = cl.VBxClustering(psi=psi).refine(rho, init)
        assert v.num_clusters == o.num_clusters and len(v.elbos) == len(o.elbos)
        assert np.abs(v.gamma - o.gamma).max() <= 1e-9 and np.abs(v.pi - o.pi).max() <= 1e-9
        assert np.abs((v.elbos - o.elbos) / o.elbos).max() <= 1e-10
        assert np.array_equal(v.hard_clusters, o.hard)
        cents = cl.compute_centroids(emb.astype(np.float64), v)
        ocents = oracle.compute_centroids(emb.astype(np.float64), o, init)
        assert cents.shape == ocents.shape and np.abs(cents - ocents).max() <= 1e-12
        labels, scores = cl.assign_embeddings(emb.astype(np.float64), cents, want_scores=True)
        olabels, oscores = oracle.assign_embeddings(emb.astype(np.float64), ocents, want_scores=True)
        assert np.array_equal(labels, olabels) and np.abs(scores - oscores).max() <= 1e-4
    # psi of the wrong length -> identity (VBxClustering.swift:71-76); no initial labels -> uniform gamma
    v = cl.VBxClustering(psi=np.ones(7)).refine(rho[:200], init[:200])
    o = oracle.vbx_refine(rho[:200], np.ones(7), init[:200])
    assert np.array_equal(v.hard_clusters, o.hard) and np.abs(v.gamma - o.gamma).max() <= 1e-9
    # run-to-run determinism (OfflineDiarizerTwoPhaseTests.swift:20-33: cluster phase bit-identical across repeats)
    a = cl.VBxClustering(psi=psi).refine(rho, init)
    b = cl.VBxClustering(psi=psi).refine(rho, init)
    assert np.array_equal(a.gamma, b.gamma) and np.array_equal(a.elbos, b.elbos)


def test_cluster_pipeline_labels_bit_exact(gpu_lib, oracle):
    for n, k, seed in ((2, 1, 0), (9, 2, 1), (500, 4, 2), (2000, 8, 3)):
        emb, _ = synth.speaker_embeddings(n, 256, k, seed=seed + 10)
        if n >= 9:
            emb[5, 3] = np.nan
            emb[n - 1, 100] = np.inf
        rho, psi = synth.synthetic_plda(np.nan_to_num(emb, posinf=0.0))
        r = cl.OfflineClusterer(psi=psi).cluster(emb, rho)
        o = oracle.diarize_cluster(emb, rho, psi, use_ref=True)
        assert np.array_equal(r.labels, o.labels), n
        assert np.array_equal(r.initial[o.training_indices], o.initial)
        assert r.info["training_count"] == o.training_indices.size
        assert r.centroids.shape == o.centroids.shape and np.abs(r.centroids - o.centroids).max() <= 1e-9
        assert r.info["detected_clusters"] == o.detected_clusters and r.info["was_adjusted"] == 0   # assignedClusterCount
    # every row non-finite -> all rows are used (selectTrainingEmbeddings, OfflineDiarizerManager.swift:606-608):
    # AHC then reports NaN and falls back to identity labels exactly like the Swift caller
    emb = np.full((6, 256), np.nan, np.float32)
    rho = np.zeros((6, 128))
    r = cl.OfflineClusterer().cluster(emb, rho)
    assert r.info["training_count"] == 6 and r.info["initial_clusters"] == 6


def test_standalone_normalise_and_linear_resample(gpu_lib, oracle):
    """fa_mel_normalize_per_feature (UnifiedMelExtractor.normalizePerFeature, time-major in place) and fa_linear_resample
    (AudioConverter.linearResample, :388-442) as standalone C-ABI calls: device kernels, bit-exact against the oracle."""
    import ctypes as C
    lib = _lib.load()
    rng = np.random.default_rng(4)
    for T, M, valid in ((6, 4, 4), (300, 80, 211), (50, 128, 50), (9, 3, 1)):
        x = (rng.standard_normal((T, M)) * 3 - 7).astype(np.float32)
        y = x.copy()
        assert lib.fa_mel_normalize_per_feature(y.ctypes.data, T, M, valid) == 0
        assert np.array_equal(y, oracle.normalize_per_feature(x, valid))
        from fluidaudio_b200 import mel as mel_mod
        assert np.array_equal(mel_mod.normalize_per_feature(x, valid), y)
    planar = np.ascontiguousarray(rng.standard_normal((3, 1000)), np.float32)
    for ch in (1, 3):
        for rin, rout in ((48000, 16000), (44100, 16000), (8000, 16000), (16000, 16000)):
            n = C.c_int64()
            p = np.ascontiguousarray(planar[:ch])
            assert lib.fa_linear_resample(p.ctypes.data, 1000, ch, rin, rout, None, 0, C.byref(n)) == 0
            out = np.zeros(n.value, np.float32)
            assert lib.fa_linear_resample(p.ctypes.data, 1000, ch, rin, rout, out.ctypes.data, out.size, C.byref(n)) == 0
            assert np.array_equal(out, oracle.linear_resample(p, rin, rout))
            assert abs(out.size - 1000 * rout / rin) <= 0.01 * 1000 * rout / rin + 1      # AudioConverterTests.swift:129-176


def test_batch_of_sets_equals_one_by_one(gpu_lib, oracle):
    sizes = [700, 1200, 300, 2, 950, 1500]
    embs, rhos, offs = [], [], [0]
    psi = None
    for i, n in enumerate(sizes):
        e, _ = synth.speaker_embeddings(n, 256, 4, weights=(0.4, 0.3, 0.2, 0.1), seed=100 + i)
        r, psi = synth.synthetic_plda(e)
        embs.append(e); rhos.append(r); offs.append(offs[-1] + n)
    c = cl.OfflineClusterer(psi=psi)
    labels, infos = c.cluster_batch(np.concatenate(embs), np.concatenate(rhos), offs)
    for i, n in enumerate(sizes):
        single = c.cluster(embs[i], rhos[i]).labels
        assert np.array_equal(labels[offs[i]:offs[i + 1]], single)
        assert np.array_equal(single, oracle.diarize_cluster(embs[i], rhos[i], psi).labels)
        assert infos[i]["training_count"] == n


def test_batch_with_chunk_indices_equals_one_by_one(gpu_lib, oracle):
    """fa_diarize_cluster_batch_chunks: the reference's default constrained assignment in every set of a batch equals the
    single-set entry point and the oracle (chunk indices are numbered inside each set)."""
    rng = np.random.default_rng(33)
    sizes = [500, 40, 900]
    embs, rhos, chunks, offs = [], [], [], [0]
    psi = None
    for i, n in enumerate(sizes):
        e, _ = synth.speaker_embeddings(n, 256, 4, weights=(0.4, 0.3, 0.2, 0.1), seed=200 + i)
        r, psi = synth.synthetic_plda(e)
        embs.append(e); rhos.append(r); offs.append(offs[-1] + n)
        chunks.append(np.sort(rng.integers(0, max(1, n // 2), n)).astype(np.int32))
    c = cl.OfflineClusterer(psi=psi)
    labels, _ = c.cluster_batch(np.concatenate(embs), np.concatenate(rhos), offs, chunk_indices=np.concatenate(chunks))
    plain, _ = c.cluster_batch(np.concatenate(embs), np.concatenate(rhos), offs)
    differs = False
    for i, n in enumerate(sizes):
        single = c.cluster(embs[i], rhos[i], chunk_indices=chunks[i]).labels
        assert np.array_equal(labels[offs[i]:offs[i + 1]], single)
        o = oracle.diarize_cluster(embs[i], rhos[i], psi, chunk_indices=chunks[i])
        assert np.array_equal(single, o.labels)
        differs |= not np.array_equal(single, plain[offs[i]:offs[i + 1]])
    assert differs   # the constraint changes at least one label on these inputs (else the test would not see the argument)
    with pytest.raises(ValueError):
        c.cluster_batch(np.concatenate(embs), np.concatenate(rhos), offs, chunk_indices=chunks[0])


def test_constrained_pipeline_matches_oracle(gpu_lib, oracle):
    """The reference's DEFAULT configuration (constrainedAssignment = true): chunk-wise Hungarian on GPU scores."""
    rng = np.random.default_rng(21)
    for n, k, seed in ((600, 4, 5), (3000, 8, 6)):
        emb, who = synth.speaker_embeddings(n, 256, k, seed=seed)
        rho, psi = synth.synthetic_plda(emb)
        chunk = np.sort(rng.integers(0, n // 2, n)).astype(np.int32)        # ~2 local speakers per chunk
        r = cl.OfflineClusterer(psi=psi).cluster(emb, rho, chunk_indices=chunk)
        o = oracle.diarize_cluster(emb, rho, psi, use_ref=True, chunk_indices=chunk)
        assert np.array_equal(r.labels, o.labels)
        plain = cl.OfflineClusterer(psi=psi).cluster(emb, rho).labels
        assert (r.labels != plain).any() or r.info["centroid_count"] == 1       # the constraint changes something
        for c in np.unique(chunk):
            a = r.labels[chunk == c]
            assert len(set(a[a >= 0].tolist())) == (a >= 0).sum()
        spk = (np.arange(n) % 3).astype(np.int32)
        m = cl.build_chunk_assignments(chunk, spk, r.labels, int(chunk.max()) + 1, 3, r.info["centroid_count"])
        assert np.array_equal(m, oracle.build_chunk_assignments(chunk, spk, o.labels, int(chunk.max()) + 1, 3,
                                                                o.centroids.shape[0]))


def test_export_replay_matches_oracle_and_file_labels(gpu_lib, oracle, tmp_path):
    """SURVEY 8f rank 2: an embedding-export file (as the reference writes it) replayed through the B200 backend gives
    the oracle's labels, and the partition stored in the file's `cluster` column is recognised."""
    from fluidaudio_b200.export_io import EmbeddingExport, PreparedDiarization, cluster_prepared
    rng = np.random.default_rng(3)
    n, k = 900, 5
    emb, _ = synth.speaker_embeddings(n, 256, k, seed=11)
    rho, psi = synth.synthetic_plda(emb)
    chunk = np.sort(rng.integers(0, n // 2, n)).astype(np.int32)
    spk = np.zeros(n, np.int32)
    for c in np.unique(chunk):                                                    # local speaker slots 0, 1, 2 ... per chunk
        idx = np.nonzero(chunk == c)[0]
        spk[idx] = np.arange(idx.size) % 3
    o = oracle.diarize_cluster(emb, rho, psi, use_ref=True, chunk_indices=chunk)
    stored = np.where(o.labels >= 0, (o.labels + 3) % (o.labels.max() + 1), o.labels).astype(np.int32)   # renamed ids
    ex = EmbeddingExport(chunk, spk, (chunk * 10).astype(np.int32), (chunk * 10 + 9).astype(np.int32),
                         chunk * 0.17, chunk * 0.17 + 0.16, emb, rho, stored)
    path = tmp_path / "meeting.json"
    ex.write(path)
    prep = PreparedDiarization.load(path)
    assert prep.embedding_count == n and prep.segmentation_chunk_count == int(chunk.max()) + 1
    rep = cluster_prepared(prep, psi)
    assert np.array_equal(rep.result.labels, o.labels)
    assert rep.matches_export is True
    assert np.array_equal(rep.chunk_assignments,
                          oracle.build_chunk_assignments(chunk, spk, o.labels, prep.num_chunks, prep.num_local_speakers,
                                                         max(int(o.labels.max()) + 1, 1)))
    plain = cluster_prepared(prep, psi, constrained=False)
    assert np.array_equal(plain.result.labels,
                          oracle.diarize_cluster(emb, rho, psi, use_ref=True).labels)


def test_mel_adapters_match_oracle(gpu_lib, oracle):
    """SURVEY 8f rank 3: UnifiedMelExtractor.features and the LS-EEND mel front end, post-processing on the GPU."""
    from fluidaudio_b200.mel import LSEENDMelFrontend, UnifiedMelExtractor
    a = synth.tone_noise_audio(16000 * 6)
    for window_samples, valid_count, n_mels in ((64000, 40000, 128), (24000, 24000, 80), (16000, 100, 128), (4800, 4000, 128)):
        window = np.zeros(window_samples, np.float32)
        window[:valid_count] = a[:valid_count]
        ex = UnifiedMelExtractor(window_samples, n_mels)
        mel, length = ex.features(window, valid_count)
        ref, valid = oracle.unified_mel_features(window, valid_count, n_mels)
        assert mel.shape == (1, n_mels, window_samples // 160 + 1) and length.tolist() == [valid]
        # the normalised value divides a log-mel difference (accurate to ~1e-6) by a std of order 1
        assert np.abs(mel[0] - ref).max() < 1e-4, (window_samples, np.abs(mel[0] - ref).max())
        assert not mel[0][:, valid:].any()
    fe = LSEENDMelFrontend()
    cfg = oracle.lseend_config()
    mean, count = np.zeros(23, np.float32), 0
    pos = 0
    # 511 samples still give one (partial) frame — Swift's (n - nFFT) / hop truncates toward zero (:345); 300 give none
    for n in (16000, 8000 + 352, 511, 300, 24000):
        chunk = a[pos:pos + n]
        pos += max(n - 352, 0)
        got = fe.process(chunk)
        if n == 300:
            assert got.shape == (0, 23) and fe.cmn_count == count
            continue
        ref, mean, count = oracle.lseend_features(cfg, chunk, mean, count)
        assert got.shape == ref.shape and fe.cmn_count == count
        assert np.abs(got - ref).max() < 1e-4
        assert np.abs(fe.cmn_mean - mean).max() < 1e-4
    fe.reset()
    assert fe.cmn_count == 0 and not fe.cmn_mean.any()


def test_kmeans_matches_oracle(gpu_lib, oracle):
    """SURVEY 8f rank 4: KMeansClustering on the GPU — labels and the winning seed exact, centroids bit-identical
    (same summation order as the oracle's restatement)."""
    six = np.array([[1.0, 0.0], [1.1, 0.1], [0.0, 1.0], [0.1, 1.1], [-1.0, 0.0], [-0.9, 0.1]])
    for emb, k, iters, seed in ((six, 3, 100, 42), (six, 1, 100, 42), (six[:2], 5, 100, 42), (six, 3, 300, 12345),
                                (np.repeat(np.eye(3), 4, axis=0), 3, 50, 1)):
        lab, cen = cl.KMeansClustering.cluster_with_centroids(emb, k, iters, seed)
        ol, oc, _ = oracle.kmeans(emb, k, iters, seed)
        assert np.array_equal(lab, ol) and cen.tobytes() == oc.tobytes()
    for n, d, k, seed in ((500, 64, 5, 9), (2000, 256, 8, 4), (300, 256, 12, 2)):
        emb, _ = synth.speaker_embeddings(n, d, min(k, 8), seed=seed)
        x = emb.astype(np.float64)
        lab, cen, best = cl.KMeansClustering.cluster_with_centroids_n_init(x, k, 100, 10, 0)
        ol, oc, ob = oracle.kmeans_ninit(x, k, 100, 10, 0)
        assert best == ob and np.array_equal(lab, ol) and cen.tobytes() == oc.tobytes()
        lab1, cen1 = cl.KMeansClustering.cluster_with_centroids(x, k, 3, 7)           # stopped by max_iterations
        ol1, oc1, _ = oracle.kmeans(x, k, 3, 7)
        assert np.array_equal(lab1, ol1) and cen1.tobytes() == oc1.tobytes()


def test_speaker_count_constraints_pipeline_matches_oracle(gpu_lib, oracle):
    """refineWithConstraints inside the pipeline: forced counts re-cluster with K-Means and skip the constrained
    assignment; satisfied constraints change nothing."""
    rng = np.random.default_rng(5)
    emb, _ = synth.speaker_embeddings(1200, 256, 5, seed=13)
    rho, psi = synth.synthetic_plda(emb)
    chunk = np.sort(rng.integers(0, 600, 1200)).astype(np.int32)
    base = cl.OfflineClusterer(psi=psi).cluster(emb, rho)
    detected = base.info["detected_clusters"]
    assert base.info["was_adjusted"] == 0 and detected >= 1
    for kw in ({"exactly": detected + 2}, {"min": detected + 1, "max": detected + 4}, {"max": max(1, detected - 1)},
               {"min": 1, "max": detected + 3}, {"exactly": -5}):
        cfg = cl.OfflineDiarizerConfig().with_speakers(**kw)
        c = cfg.clustering
        for chunks in (None, chunk):
            r = cl.OfflineClusterer(cfg, psi=psi).cluster(emb, rho, chunk_indices=chunks)
            o = oracle.diarize_cluster(emb, rho, psi, use_ref=True, chunk_indices=chunks,
                                       num_speakers=c.num_speakers, min_speakers=c.min_speakers, max_speakers=c.max_speakers)
            assert bool(r.info["was_adjusted"]) == o.was_adjusted and r.info["detected_clusters"] == o.detected_clusters
            assert np.array_equal(r.labels, o.labels), kw
            assert r.centroids.shape == o.centroids.shape and np.abs(r.centroids - o.centroids).max() < 1e-12


def test_vbx_with_hundreds_and_thousands_of_speakers(gpu_lib, oracle):
    """Degenerate AHC output (every embedding nearly its own cluster) must still run: the E-step reads alpha through L2
    when S x D x 8 exceeds shared memory, and beyond 1 024 speakers the partial sums use fewer frame chunks."""
    for T, S, D in ((600, 260, 128), (1300, 1100, 64)):
        rng = np.random.default_rng(S)
        emb, _ = synth.speaker_embeddings(T, 256, 6, seed=S)
        rho, psi = synth.synthetic_plda(emb, D)
        init = np.concatenate([np.arange(S), rng.integers(0, S, T - S)]).astype(np.int32)   # every label occurs
        g = cl.VBxClustering(psi=psi).refine(rho, init)
        o = oracle.vbx_refine(rho, psi, init)
        assert g.gamma.shape == (T, S) and g.elbos.size == o.elbos.size
        assert np.abs(g.elbos - o.elbos).max() <= 1e-9 * np.abs(o.elbos).max()
        assert np.abs(g.gamma - o.gamma).max() < 1e-8 and np.abs(g.pi - o.pi).max() < 1e-10
        cents = cl.compute_centroids(emb.astype(np.float64), g)
        ocents = oracle.compute_centroids(emb.astype(np.float64), o, init)
        assert cents.shape == ocents.shape and np.abs(cents - ocents).max() < 1e-9
    # the whole phase with a threshold that leaves ~hundreds of clusters to VBx
    emb, _ = synth.speaker_embeddings(500, 256, 4, seed=77)
    rho, psi = synth.synthetic_plda(emb)
    cfg = cl.OfflineDiarizerConfig()
    cfg.clustering.threshold = 0.2
    r = cl.OfflineClusterer(cfg, psi=psi).cluster(emb, rho)
    o = oracle.diarize_cluster(emb, rho, psi, threshold=0.2, use_ref=True)
    assert r.info["initial_clusters"] == len(set(o.initial.tolist())) and r.info["initial_clusters"] > 200
    assert r.info["vbx_iterations"] == o.vbx.elbos.size and r.centroids.shape == o.centroids.shape
    assert np.abs(r.centroids - o.centroids).max() < 1e-9


def test_next_rows_against_committed_goldens(gpu_lib, golden_dir):
    """CUDA path vs tests/golden/next_rows.npz (made by tests/golden/make_golden.py): nothing of the oracle runs here."""
    import os
    from fluidaudio_b200.mel import LSEENDMelFrontend, UnifiedMelExtractor
    g = np.load(os.path.join(golden_dir, "next_rows.npz"))
    six = np.array([[1.0, 0.0], [1.1, 0.1], [0.0, 1.0], [0.1, 1.1], [-1.0, 0.0], [-0.9, 0.1]])
    for name, (k, iters, seed) in {"six_k3_seed42": (3, 100, 42), "six_k3_seed12345": (3, 300, 12345)}.items():
        lab, cen = cl.KMeansClustering.cluster_with_centroids(six, k, iters, seed)
        assert np.array_equal(lab, g[f"kmeans_{name}__labels"]) and cen.tobytes() == g[f"kmeans_{name}__centroids"].tobytes()
    emb, _ = synth.speaker_embeddings(300, 64, 5, seed=9)
    lab, cen, best = cl.KMeansClustering.cluster_with_centroids_n_init(emb.astype(np.float64), 5, 100, 10, 0)
    assert best == int(g["kmeans_ninit_300x64__best"][0]) and np.array_equal(lab, g["kmeans_ninit_300x64__labels"])
    assert cen.tobytes() == g["kmeans_ninit_300x64__centroids"].tobytes()
    a = synth.tone_noise_audio(16000)
    mel, length = UnifiedMelExtractor(8000).features(np.concatenate([a[:6000], np.zeros(2000, np.float32)]), 6000)
    assert length.tolist() == g["unified_8000_valid6000__valid"].tolist()
    assert np.abs(mel[0] - g["unified_8000_valid6000__mel"]).max() < 1e-4
    fe = LSEENDMelFrontend()
    f1 = fe.process(a[:4000])
    f2 = fe.process(a[4000 - 352:9000])
    assert np.abs(f1 - g["lseend__f1"]).max() < 1e-4 and np.abs(f2 - g["lseend__f2"]).max() < 1e-4
    assert np.abs(fe.cmn_mean - g["lseend__mean"]).max() < 1e-4 and fe.cmn_count == int(g["lseend__count"][0])


def test_pipeline_odd_shapes_and_tiny_inputs(gpu_lib, oracle):
    """Shapes the fuzz sweep (scripts/gpu_fuzz.py) covers, pinned as a test: embedding widths that are not 256, one to five
    embeddings, filtered (NaN / Inf) rows, a PLDA vector of the wrong length (-> identity, VBxClustering.swift:71-76).
    Labels must agree wherever the decision is not a rounding-level tie (two identical centroids can come out of VBx)."""
    rng = np.random.default_rng(12)
    cases = [(1, 256, 1), (2, 256, 2), (3, 64, 2), (5, 192, 2), (17, 64, 2), (100, 255, 3), (333, 257, 3), (400, 192, 4)]
    for n, d, k in cases:
        emb, _ = synth.speaker_embeddings(n, d, k, seed=n + d)
        if n >= 100:
            emb[rng.integers(0, n)] = np.nan
            emb[rng.integers(0, n)] = np.inf
        rho, psi = synth.synthetic_plda(np.nan_to_num(emb, nan=0.0, posinf=0.0, neginf=0.0), min(128, d))
        for p in (psi, psi[:-1]):                                   # second pass: wrong length -> identity on both sides
            got = cl.OfflineClusterer(psi=p).cluster(emb, rho)
            ref = oracle.diarize_cluster(emb, rho, p, use_ref=True)
            assert got.info["training_count"] == ref.training_indices.size
            assert np.array_equal(got.initial[got.initial >= 0], ref.initial)
            assert got.centroids.shape == ref.centroids.shape and np.abs(got.centroids - ref.centroids).max() < 1e-9
            ok = np.isfinite(emb).all(axis=1)
            cn = ref.centroids / np.maximum(np.linalg.norm(ref.centroids, axis=1, keepdims=True), 1e-300)
            e = np.where(ok[:, None], emb, 0.0).astype(np.float64)
            sc = (e / np.maximum(np.linalg.norm(e, axis=1, keepdims=True), 1e-300)) @ cn.T
            srt = np.sort(sc, axis=1)
            decided = ok & ((srt[:, -1] - srt[:, -2] > 1e-9) if sc.shape[1] > 1 else np.ones(n, bool))
            assert np.array_equal(got.labels[decided], ref.labels[decided]), (n, d, k)
