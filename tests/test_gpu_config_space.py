"""The log-mel kernels and the resampler across the configurations the library accepts, against the float64 oracle
(run with ``-m gpu`` on the B200 box).

tests/test_gpu_parity.py checks the front end mostly at the benchmark's shape (hop 160, win 400, 80 / 128 mels, 16 kHz).
Here every value of every axis below runs with both transform precisions and through ``compute_flat_transposed``
(time-major), ``compute_flat`` (mel-major) and legacy ``compute()``, on lengths chosen so that frame counts land on,
just past and just short of the 16-frame tile (T mod 16 in {0, 1, 15}), below one tile, and on every sample count
mod 4 (the kernel's 16-byte staging), plus clips shorter than half a frame.

Bars:
  * FP64 transform: |log-mel - oracle| <= MEL_TOL (1e-4);
  * float32 transform: max |delta| of a call within max(1e-4, 2 max |oracle(float32 FFT) - oracle|), i.e. no worse than
    twice an independent float32 FFT (oracle precision 2) on the same input (floor 5e-4 without pre-emphasis);
  * shapes, frame counts and non-finite values: exact.
The largest |delta| of each path is printed (``-s``).
"""
import numpy as np
import pytest

from fluidaudio_b200 import _lib, synth
from fluidaudio_b200.audio_converter import AudioConverter
from fluidaudio_b200.mel import AudioMelSpectrogram, LogFloorMode, PaddingMode, Precision

pytestmark = pytest.mark.gpu

MEL_TOL = 1e-4
# Without pre-emphasis (legacy compute(), preemph 0) a frame keeps its full dynamic range and the float32 transform's
# noise floor shows in weak bins at up to ~4e-4, where an independent float32 FFT can happen to land closer
F32_FLOOR_NO_PREEMPH = 5e-4

BASE = dict(sample_rate=16000, n_mels=80, n_fft=512, hop_length=160, win_length=400, preemph=0.97, pad_to=1,
            log_floor=2.0 ** -24, log_floor_mode=0, window_periodic=False)

HOPS = [2, 4, 6, 14, 80, 158, 160, 162, 256, 320, 510, 512, 514, 640, 676, 677, 678, 679, 680, 800, 862, 863, 864,
        865, 866, 888, 889, 890, 891, 892, 1000, 1022, 1024]
HOPS_GENERIC = [161, 1026]                     # odd hop and hop > 1024: the any-nFFT kernel (routing controls)
WINS = [2, 31, 64, 255, 256, 320, 383, 384, 399, 400, 401, 447, 448, 449, 511, 512]
N_MELS = [1, 2, 3, 4, 5, 23, 40, 81, 127, 128, 129, 256, 257, 512]
RATES = [8000, 16000, 22050, 24000, 44100, 48000]
PREEMPHS = [0.97, 0.0, -0.5]
FLOORS = [(mode, fl) for mode in (0, 1) for fl in (2.0 ** -24, 1e-10, 1e-38)]

_max_delta = {}


def _note(path, d):
    _max_delta[path] = max(_max_delta.get(path, 0.0), float(d))


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    for path in sorted(_max_delta):
        print(f"\nmax |delta| {path}: {_max_delta[path]:.3e}", end="")
    print()


# ------------------------------------------------------------------------------------------------ signals
def _square(n, sr):
    t = np.arange(n) / sr
    return np.where(np.sin(2 * np.pi * 310.0 * t) >= 0, 1.0, -1.0).astype(np.float32)


def _tiny_noise(n, sr):
    return (1e-6 * np.random.default_rng(n).standard_normal(n)).astype(np.float32)


def _dc(n, sr):
    return (0.5 + synth.tone_noise_audio(n, seed=3, sample_rate=sr) * np.float32(0.01)).astype(np.float32)


def _silent_middle(n, sr):
    a = synth.speech_like_audio(n, sample_rate=sr)
    a[n // 4: 3 * n // 4] = 0.0
    return a


SIGNALS = {
    "tone_noise": lambda n, sr: synth.tone_noise_audio(n, seed=n % 13, sample_rate=sr),
    "speech_like": lambda n, sr: synth.speech_like_audio(n, sample_rate=sr),
    "square": _square,
    "noise_1e-6": _tiny_noise,
    "dc": _dc,
    "silent_middle": _silent_middle,
    "zeros": lambda n, sr: np.zeros(n, np.float32),
}


def _length(cfg, frames, mod4):
    """A sample count whose centre-mode frame count is `frames` (or the smallest possible) and whose value mod 4 is
    `mod4` wherever the hop leaves room for it."""
    hop, win = cfg["hop_length"], cfg["win_length"]
    n = max(1, (frames - 1) * hop + win - cfg["n_fft"])
    span = min(hop, 4)
    for r in range(span):
        if (n + r) % 4 == mod4:
            return n + r
    return n


# ------------------------------------------------------------------------------------------------ comparison
def _oracle_cfg(oracle, cfg, precision=0):
    kw = dict(cfg)
    kw["window_periodic"] = int(bool(kw["window_periodic"]))
    return oracle.mel_config(precision=precision, **kw)


def _compare(path, got, ref, ref32=None, ctx=(), f32_floor=MEL_TOL):
    """ref: oracle (precision 0); ref32: oracle with a float32 FFT, given for the float32 transform."""
    got = np.asarray(got, np.float32).reshape(ref.shape)
    fin = np.isfinite(ref)
    assert np.array_equal(np.isfinite(got), fin), (path, ctx)
    assert np.array_equal(got[~fin], ref[~fin]), (path, ctx)        # -inf where the oracle has -inf
    d = np.where(fin, np.abs(got.astype(np.float64) - np.where(fin, ref, 0.0)), 0.0)
    if d.size:
        _note(path, d.max())
    if ref32 is None:
        assert d.max() <= MEL_TOL, (path, ctx, float(d.max()))
    else:
        # float32 transform noise is ~0.5 ulp of a frame's largest line in every bin and lands differently in every FFT:
        # the worst element of the call within twice the worst departure of an independent float32 FFT on the same input
        spread = np.where(fin, np.abs(np.where(fin, ref32, 0.0).astype(np.float64) - np.where(fin, ref, 0.0)), 0.0)
        bar = max(f32_floor, 2.0 * float(spread.max()))
        assert d.max() <= bar, (path, ctx, float(d.max()), bar)


def _check_config(oracle, cfg, sig_name, n, entry=0, last=0.0, tag=""):
    """Every entry point of one configuration, both precisions, against the oracle.  entry rotates the padding mode of
    the time-major call: 0 centre, 1 prePadded, 2 prePadded with fewer frames expected, 3 with more."""
    sr = cfg["sample_rate"]
    a = SIGNALS[sig_name](n, sr)
    o0, o2 = _oracle_cfg(oracle, cfg, 0), _oracle_cfg(oracle, cfg, 2)
    nm = cfg["n_mels"]
    mode = PaddingMode.center if entry == 0 else PaddingMode.pre_padded
    natural = oracle.mel_frame_count(o0, n, int(mode))
    expected = {0: None, 1: None, 2: max(1, natural - 3), 3: natural + 17}[entry]
    refs = {
        "flat_transposed": oracle.mel_flat_transposed(o0, a, last=last, padding_mode=int(mode), expected_frames=expected),
        "flat": oracle.mel_flat(o0, a, last=last),
        "legacy": oracle.mel_legacy(o0, a),
    }
    refs32 = {
        "flat_transposed": oracle.mel_flat_transposed(o2, a, last=last, padding_mode=int(mode), expected_frames=expected),
        "flat": oracle.mel_flat(o2, a, last=last),
        "legacy": oracle.mel_legacy(o2, a),
    }
    kw = dict(cfg)
    kw["log_floor_mode"] = LogFloorMode(kw["log_floor_mode"])
    floor32 = MEL_TOL if cfg["preemph"] != 0.0 else F32_FLOOR_NO_PREEMPH
    for prec in (Precision.f64, Precision.f32):
        m = AudioMelSpectrogram(precision=prec, **kw)
        where = f"{prec.name}"
        ctx = (tag, sig_name, n, entry, prec.name)
        r32 = (lambda k: refs32[k][0]) if prec == Precision.f32 else (lambda k: None)
        got, ml, nf = m.compute_flat_transposed(a, last_audio_sample=last, padding_mode=mode, expected_frame_count=expected)
        ref, rml, rnf = refs["flat_transposed"]
        assert (ml, nf) == (rml, rnf) and got.size == nf * nm, ctx
        _compare(f"{where}/time-major", got, ref, r32("flat_transposed"), ctx, floor32)
        got, ml, nf = m.compute_flat(a, last_audio_sample=last)
        ref, rml, rnf = refs["flat"]
        assert (ml, nf) == (rml, rnf) and got.size == nf * nm, ctx
        _compare(f"{where}/mel-major", got, ref, r32("flat"), ctx, floor32)
        got, ml = m.compute(a)
        ref, rml = refs["legacy"]
        assert ml == rml, ctx
        if ml:
            assert got.shape == (1, nm, ml), ctx
            _compare(f"{where}/legacy", got[0], ref, r32("legacy"), ctx, F32_FLOOR_NO_PREEMPH)
        m.close()


_FRAMES = [32, 33, 31, 5]                          # T mod 16 = 0, 1, 15 and T < 16
_SIGS = [s for s in SIGNALS if s != "zeros"]   # all-zero input runs with the floors that matter for it


def _axis_cases():
    cases = []
    axes = [("hop_length", HOPS + HOPS_GENERIC), ("win_length", WINS), ("n_mels", N_MELS), ("sample_rate", RATES),
            ("preemph", PREEMPHS)]
    for name, values in axes:
        for v in values:
            for periodic in ((False, True) if name == "win_length" else (False,)):
                cases.append((f"{name}={v}" + (" periodic" if periodic else ""), {name: v, "window_periodic": periodic}))
    for mode, fl in FLOORS:
        cases.append((f"floor {'clamped' if mode else 'additive'} {fl:g}", {"log_floor_mode": mode, "log_floor": fl}))
    for p in (1, 3, 16):
        cases.append((f"pad_to={p}", {"pad_to": p}))
    cases.append(("nFFT=1024 hop=160", {"n_fft": 1024}))
    return cases


@pytest.mark.parametrize("tag,over", _axis_cases(), ids=[c[0] for c in _axis_cases()])
def test_mel_axis_against_oracle(gpu_lib, oracle, tag, over):
    """One axis value away from the default configuration, on two signals / lengths / padding modes from the rotation."""
    cfg = dict(BASE, **over)
    i = sum(map(ord, tag))                                            # deterministic rotation index
    for j in range(2):
        k = i + j
        n = _length(cfg, _FRAMES[k % 4], k % 4)
        _check_config(oracle, cfg, _SIGS[k % len(_SIGS)], n, entry=k % 4, last=(0.0, 0.3, -0.7)[k % 3], tag=tag)


def test_mel_short_clips_every_axis(gpu_lib, oracle):
    """Clips shorter than half a frame (n < nFFT / 2, one partially filled centre frame) on a spread of configurations."""
    for j, over in enumerate([{}, {"hop_length": 2}, {"hop_length": 1024}, {"win_length": 31}, {"n_mels": 512},
                              {"n_mels": 1}, {"preemph": -0.5}, {"win_length": 512, "window_periodic": True}]):
        cfg = dict(BASE, **over)
        for n in (1, 2, 3, 4, 100, 255):
            _check_config(oracle, cfg, _SIGS[(j + n) % len(_SIGS)], n, entry=(j + n) % 2, last=0.25, tag=str(over))


@pytest.mark.parametrize("hop", HOPS)
def test_mel_hop_by_window_grid(gpu_lib, oracle, hop):
    """Pairwise hop x window at 80 mels: every tile geometry (scalar / vector pre-emphasis, staged span) meets every
    window placement (centred pass 1 with and without the full middle, legacy offset 0)."""
    for w, win in enumerate(WINS):
        cfg = dict(BASE, hop_length=hop, win_length=win, window_periodic=bool(w & 1))
        k = w + hop
        _check_config(oracle, cfg, _SIGS[k % len(_SIGS)], _length(cfg, _FRAMES[k % 4], k % 4), entry=k % 4,
                      last=0.1 * (k % 3), tag=f"hop={hop} win={win}")


@pytest.mark.parametrize("sample_rate", RATES)
def test_mel_n_mels_by_sample_rate_grid(gpu_lib, oracle, sample_rate):
    for j, nm in enumerate(N_MELS):
        cfg = dict(BASE, sample_rate=sample_rate, n_mels=nm)
        _check_config(oracle, cfg, _SIGS[j % len(_SIGS)], _length(cfg, _FRAMES[j % 4], j % 4), entry=j % 4,
                      tag=f"sr={sample_rate} n_mels={nm}")


def test_mel_all_zero_input_and_non_finite_floors(gpu_lib, oracle):
    """Silence with a floor below the smallest normal float (the kernel's denormal log path) and with floor 0 (-inf)."""
    for mode in (0, 1):
        for fl in (1e-38, 0.0):
            for over in ({}, {"hop_length": 162, "win_length": 255}, {"n_mels": 257}):
                cfg = dict(BASE, log_floor=fl, log_floor_mode=mode, **over)
                for n in (3, _length(cfg, 33, 1)):
                    _check_config(oracle, cfg, "zeros", n, entry=n % 4, tag=f"zeros floor {fl}")


def test_mel_n_mels_513_is_rejected(gpu_lib):
    with pytest.raises(_lib.FluidAudioError) as e:
        AudioMelSpectrogram(n_mels=513)
    assert e.value.status == 8


def test_mel_long_hops_construct_and_take_the_any_nfft_kernel(gpu_lib, oracle):
    """Even hops up to 1024 with nFFT 512 whose specialised tile (15 hops + 512 samples, staged three times) exceeds the
    per-CTA shared memory must still construct and compute the oracle's values, at the largest mel count too."""
    for nm in (80, 128, 512):
        for hop in (676, 680, 864, 890, 1000, 1024):
            cfg = dict(BASE, n_mels=nm, hop_length=hop)
            _check_config(oracle, cfg, "tone_noise", _length(cfg, 17, hop % 4), entry=1, tag=f"n_mels={nm} hop={hop}")


# ------------------------------------------------------------------------------------------------ consistency
def test_mel_batch_equals_one_by_one(gpu_lib):
    """compute_batch == compute_flat_transposed / compute_flat clip by clip, bitwise, with clips whose frame counts end one
    frame into a tile next to each other (a tile never mixes two clips)."""
    for prec in (Precision.f64, Precision.f32):
        for over in ({}, {"hop_length": 162, "win_length": 255}, {"n_mels": 5, "hop_length": 2}, {"n_mels": 1},
                     {"hop_length": 890}, {"hop_length": 161}):
            cfg = dict(BASE, **over)
            m = AudioMelSpectrogram(precision=prec, **cfg)
            lens = [_length(cfg, f, r) for f, r in ((33, 1), (17, 2), (49, 3), (1, 0), (16, 1), (32, 2))] + [3, 0]
            clips = [synth.speech_like_audio(n, seed=i) if n else np.zeros(0, np.float32) for i, n in enumerate(lens)]
            last = np.linspace(-0.3, 0.3, len(clips)).astype(np.float32)
            for time_major in (True, False):
                out, offs, ml, nf = m.compute_batch(clips, last_samples=last, time_major=time_major)
                for i, c in enumerate(clips):
                    if time_major:
                        single, sml, snf = m.compute_flat_transposed(c, last_audio_sample=float(last[i]))
                    else:
                        single, sml, snf = m.compute_flat(c, last_audio_sample=float(last[i]))
                    assert (ml[i], nf[i]) == (sml, snf), (over, i)
                    assert np.array_equal(out[offs[i]:offs[i + 1]], single), (prec.name, over, time_major, i)
            m.close()


def test_mel_device_entry_with_unaligned_input(gpu_lib):
    """compute_device reading from a pointer 4 bytes past a 16-byte boundary (no bulk copies) == the host entry point."""
    for prec in (Precision.f64, Precision.f32):
        for over in ({}, {"hop_length": 162, "win_length": 255}, {"n_mels": 3, "hop_length": 6}, {"hop_length": 1024}):
            cfg = dict(BASE, **over)
            m = AudioMelSpectrogram(precision=prec, **cfg)
            a = synth.tone_noise_audio(_length(cfg, 65, 3))
            T = m.frame_count(a.size)
            host, _, _ = m.compute_flat_transposed(a, last_audio_sample=0.2)
            d_a = _lib.DeviceBuffer(a.nbytes + 64)
            d_o = _lib.DeviceBuffer(T * cfg["n_mels"] * 4)
            d_a.upload(np.concatenate([np.zeros(1, np.float32), a]))

            class Off:
                ptr = d_a.ptr.value + 4
            assert m.compute_device(Off, a.size, d_o, last_audio_sample=0.2) == (T, T)
            _lib.synchronize()
            assert np.array_equal(d_o.download((T * cfg["n_mels"],), np.float32), host), (prec.name, over)
            m.close()


def test_mel_unaligned_outputs(gpu_lib):
    """Outputs that are not 16-byte aligned: a device pointer 4 bytes into a buffer, batch output offsets that are not
    multiples of four floats and a pinned host view one float in, stored through by the kernel (zero-copy).  Rows of
    n_mels % 4 == 0 must then be stored one float at a time; the values equal the aligned call's."""
    m = AudioMelSpectrogram(n_mels=80)
    a = synth.tone_noise_audio(16000 * 3 + 5)
    T = m.frame_count(a.size)
    host, _, _ = m.compute_flat_transposed(a)
    d_a = _lib.DeviceBuffer(a.nbytes + 64)
    d_a.upload(a)
    d_o = _lib.DeviceBuffer(T * 80 * 4 + 64)

    class OutOff:
        ptr = d_o.ptr.value + 4
        nbytes = T * 80 * 4
    assert m.compute_device(d_a, a.size, OutOff) == (T, T)
    _lib.synchronize()
    assert np.array_equal(d_o.download((T * 80 + 1,), np.float32)[1:], host)
    # batch on the device, clip i's output at 1 + i floats past its packed position
    clips = [a[:5000], a[:16000], a[:331]]
    packed = np.concatenate(clips)
    offs = np.array([0, 5000, 21000, 21331], np.int64)
    Ts = [m.frame_count(c.size) for c in clips]
    out_offs = np.zeros(4, np.int64)
    for i in range(3):
        out_offs[i + 1] = out_offs[i] + Ts[i] * 80 + 1
    out_offs[:3] += 1
    d_p = _lib.DeviceBuffer(packed.nbytes)
    d_p.upload(packed)
    d_b = _lib.DeviceBuffer(int(out_offs[-1] + 8) * 4)
    ml, nf = m.compute_batch_device(d_p, offs, d_b, out_offs)
    _lib.synchronize()
    flat = d_b.download((int(out_offs[-1] + 8),), np.float32)
    for i, c in enumerate(clips):
        single, _, _ = m.compute_flat_transposed(c)
        assert (ml[i], nf[i]) == (Ts[i], Ts[i]) and np.array_equal(flat[out_offs[i]:out_offs[i] + Ts[i] * 80], single), i
    # zero-copy pinned output one float into the allocation: long enough for the chunked pipeline
    n = 16000 * 100
    b = synth.tone_noise_audio(n)
    Tb = m.frame_count(n)
    ref, _, _ = m.compute_flat_transposed(b)
    ref16, _, _, _ = m.compute_from_pcm(b, 48000.0)
    pin = _lib.PinnedArray(Tb * 80 + 1, np.float32)
    _lib.check(m._L.fa_mel_set_zero_copy_output(m._h, 1), "zero copy")
    pin.array[:] = -1.0
    got, ml, nf = m.compute_flat_transposed(b, out=pin.array[1:])
    assert (ml, nf) == (Tb, Tb) and np.array_equal(got, ref)
    pin.array[:] = -1.0
    got, ml, nf, _ = m.compute_from_pcm(b, 48000.0, out=pin.array[1:])
    assert np.array_equal(got, ref16)
    pin.free()
    m.close()


# ------------------------------------------------------------------------------------------------ resampler
def _sine_pcm(rate, channels, seconds, seed=0):
    rng = np.random.default_rng(seed)
    t = np.arange(int(rate * seconds)) / rate
    return np.stack([(0.5 * np.sin(2 * np.pi * (440.0 + 110.0 * c) * t) + 0.01 * rng.standard_normal(t.size)).astype(np.float32)
                     for c in range(channels)])


INT_RATES = [8000, 11025, 12000, 16001, 22050, 24000, 44101, 47999, 96000, 192000]
FRAC_RATES = [22050.25, 44100.5, 44100.001, 47999.999, 48000.001, 16000.001]


def _rs_bar(oracle, rate, target):
    L, _, _, _ = oracle.sinc_design(rate, target)
    return 3e-6 if L <= 2048 else 2e-5               # exact-phase table / interpolated between 1024 phases


@pytest.mark.parametrize("rate", INT_RATES + FRAC_RATES)
def test_resampler_against_the_float64_filter(gpu_lib, oracle, rate):
    for target in (16000, 8000):
        x = _sine_pcm(rate, 1, 0.35, seed=int(rate))[0]
        got = AudioConverter(sample_rate=target).resample(x, rate)
        ref = oracle.sinc_resample(x, rate, target)
        assert got.shape == ref.shape, (rate, target)
        d = np.abs(got.astype(np.float64) - ref).max()
        _note(f"resample {'exact' if _rs_bar(oracle, rate, target) < 1e-5 else 'interpolated'}", d)
        assert d <= _rs_bar(oracle, rate, target), (rate, target, d)
    # 8 kHz model rate through the fused PCM -> log-mel pipeline: bitwise the two-step path, and near the oracle chain
    m = AudioMelSpectrogram(sample_rate=8000, n_mels=40)
    x = _sine_pcm(rate, 1, 1.0, seed=7)[0]
    mono = AudioConverter(sample_rate=8000).resample(x, rate)
    ref, rml, rnf = m.compute_flat_transposed(mono)
    got, ml, nf, rs = m.compute_from_pcm(x, rate)
    assert (ml, nf, rs) == (rml, rnf, mono.size) and np.array_equal(got, ref), rate
    chain, cml, _ = oracle.mel_flat_transposed(oracle.mel_config(sample_rate=8000, n_mels=40), oracle.sinc_resample(x, rate, 8000))
    assert cml == ml and np.abs(got.reshape(nf, 40) - chain).max() <= 2e-3
    m.close()


def test_resampler_long_input_far_end(gpu_lib, oracle):
    """10 min of 44.1 kHz audio: output indices reach 9.6e6, i * M passes 2^31 at i ~ 4.87e6.  Windows at the start,
    across that index and at the end against the windowed oracle; the chunked PCM -> log-mel pipeline equals the
    two-step path bitwise over the whole clip."""
    rate = 44100
    x = _sine_pcm(rate, 1, 600.5, seed=3)[0]
    conv = AudioConverter()
    y = conv.resample(x, rate)
    assert y.size == oracle.resample_output_count(x.size, rate, 16000)
    _, M, _, _ = oracle.sinc_design(rate, 16000)
    cross = (1 << 31) // M
    for first in (0, cross - 3000, y.size - 6000):
        ref = oracle.sinc_resample(x, rate, 16000, first=first, count=6000)
        d = np.abs(y[first:first + 6000].astype(np.float64) - ref).max()
        _note("resample long input", d)
        assert d <= 3e-6, (first, d)
    m = AudioMelSpectrogram(n_mels=80)
    ref, rml, rnf = m.compute_flat_transposed(y)
    got, ml, nf, rs = m.compute_from_pcm(x, rate)
    assert (ml, nf, rs) == (rml, rnf, y.size) and np.array_equal(got, ref)
    # a fractional rate over a minute: every CTA's phase sums exceed 32 bits
    xf = _sine_pcm(44100.001, 1, 60.0, seed=4)[0]
    yf = conv.resample(xf, 44100.001)
    for first in (0, yf.size // 2, yf.size - 3000):
        ref = oracle.sinc_resample(xf, 44100.001, 16000, first=first, count=3000)
        assert np.abs(yf[first:first + 3000].astype(np.float64) - ref).max() <= 2e-5, first
    m.close()


def test_int16_full_scale_stereo_interleaved_equals_planar(gpu_lib, oracle):
    """int16 at exactly -32768 and 32767: the interleaved-stereo fast path (one 32-bit load per frame) == planar == the
    oracle's mixdown at the model rate, bitwise; and interleaved == planar through the resampler."""
    rng = np.random.default_rng(9)
    n = 40000
    p = rng.integers(-32768, 32768, size=(2, n)).astype(np.int16)
    p[0, :64] = np.array([-32768, 32767] * 32, np.int16)             # every pairing of the two extremes
    p[1, :64] = np.array([-32768, -32768, 32767, 32767] * 16, np.int16)
    inter = np.ascontiguousarray(p.T)
    assert (p == -32768).any() and (p == 32767).any()
    for rate in (16000, 44100, 44100.001):
        conv = AudioConverter()
        a = conv.resample_buffer(inter, rate, interleaved=True)
        b = conv.resample_buffer(p, rate)
        assert np.array_equal(a, b), rate
        if rate == 16000:
            assert np.array_equal(a, oracle.mixdown(p))
        else:
            assert np.abs(a.astype(np.float64) - oracle.sinc_resample(oracle.mixdown(p), rate, 16000)).max() <= _rs_bar(oracle, rate, 16000)
