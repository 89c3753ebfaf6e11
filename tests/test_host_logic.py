"""CPU tests of the product's host side (no GPU needed, no compute calls into the CUDA library):

* the C-ABI library loads and exports every symbol the public headers declare;
* argument contracts that are decided before any device work (the reference's own status codes);
* "no CPU fallback": without a B200 every compute entry point fails loudly;
* the product never touches oracle/;
* the device code's per-lane FFT / mel math and the merge kernel's control plane, compiled for the host from the
  SAME headers the kernels use (tests/emul/*.cpp), against the oracle and the reference goldens;
* sharding helpers, including a 2-rank gloo run.
"""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from fluidaudio_b200 import _lib, sharding, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_lib.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    return _lib.load()


def _declared_functions(header):
    text = open(os.path.join(ROOT, "include", header)).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return set(re.findall(r"\b(fa_[a-z0-9_]+|fastcluster_compute_centroid_linkage)\s*\(", text))


def test_library_exports_every_declared_symbol(lib):
    declared = _declared_functions("fluidaudio_b200.h") | _declared_functions("FastClusterWrapper.h")
    assert "fastcluster_compute_centroid_linkage" in declared and len(declared) >= 35
    out = subprocess.check_output(["nm", "-D", "--defined-only", _lib.LIB_PATH], text=True)
    exported = {line.split()[-1] for line in out.splitlines() if " T " in line}
    assert declared <= exported, f"declared but not exported: {sorted(declared - exported)}"
    assert set(_lib.EXPORTED_SYMBOLS) == declared
    # nothing but the C ABI leaks out of the shared object
    assert all(s.startswith("fa_") or s.startswith("fastcluster_") for s in exported), sorted(exported)[:10]


def test_ahc_placement_diagnostic_is_zero_before_any_linkage(lib):
    """fa_ahc_last_placement reports the calling thread's last linkage: a fresh thread sees zeros, without a device."""
    import threading
    seen = []

    def read():
        out = np.full(6, -1, np.int32)
        lib.fa_ahc_last_placement(out.ctypes.data)
        seen.append(out.tolist())

    t = threading.Thread(target=read)
    t.start()
    t.join()
    assert seen == [[0] * 6]
    lib.fa_ahc_last_placement(None)   # a null output is ignored


def test_reference_argument_contract_needs_no_device(lib):
    """FastClusterWrapper.cpp:203-223 — these statuses are decided before any clustering work."""
    f = lib.fastcluster_compute_centroid_linkage
    x = np.ones((3, 2))
    z = np.zeros(8)
    assert f(None, 3, 2, z.ctypes.data, 8) == 1
    assert f(x.ctypes.data, 3, 2, None, 8) == 1
    assert f(x.ctypes.data, 0, 2, z.ctypes.data, 8) == 0
    assert f(x.ctypes.data, 3, 0, z.ctypes.data, 8) == 1
    assert f(x.ctypes.data, 2 ** 31, 2, z.ctypes.data, 8) == 2
    assert f(x.ctypes.data, 3, 2 ** 31, z.ctypes.data, 8) == 2
    assert f(x.ctypes.data, 3, 2, z.ctypes.data, 7) == 3
    assert f(x.ctypes.data, 1, 2, z.ctypes.data, 0) == 0
    assert np.all(z == 0)


def test_swift_level_guards_need_no_device(lib):
    from fluidaudio_b200.clustering import AHCClustering
    ahc = AHCClustering()
    assert ahc.cluster([], 0.7).size == 0                                   # AHCClusteringTests.swift:12-15
    assert ahc.cluster(np.zeros((3, 0)), 0.7).tolist() == [0, 0, 0]         # :137-145
    labels = np.zeros(1, np.int32)
    assert lib.fa_ahc_cluster(np.ones((1, 3)).ctypes.data, 1, 3, 0.7, labels.ctypes.data) == 0 and labels[0] == 0


def test_no_cpu_fallback_without_a_device(lib):
    if _lib.device_count() > 0:
        pytest.skip("a B200 is visible here; the no-device behaviour is exercised on CPU-only boxes")
    from fluidaudio_b200.mel import AudioMelSpectrogram
    from fluidaudio_b200.clustering import OfflineClusterer, centroid_linkage
    with pytest.raises(_lib.FluidAudioError) as e:
        AudioMelSpectrogram()
    assert e.value.status == 6 and "no CPU fallback" in str(e.value)
    emb, _ = synth.speaker_embeddings(50, 16, 2)
    with pytest.raises(_lib.FluidAudioError):
        OfflineClusterer().cluster(emb, emb.astype(np.float64))
    st, _ = centroid_linkage(np.eye(3))
    assert st == 5      # the Swift caller maps a non-zero status to identity labels (AHCClustering.swift:52-55)


def test_product_never_imports_or_links_the_oracle():
    pkg = os.path.join(ROOT, "fluidaudio_b200")
    for dirpath, _, files in os.walk(pkg):
        for name in files:
            if name.endswith((".py", ".cu", ".cuh", ".h", ".cpp")) or name == "Makefile":
                text = open(os.path.join(dirpath, name), errors="ignore").read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", text, re.M), f"{name} imports oracle"
                assert "liboracle" not in text and "oracle_" not in text, f"{name} references the oracle"
    out = subprocess.check_output(["ldd", _lib.LIB_PATH], text=True)
    assert "oracle" not in out


def test_helpers_that_run_on_the_host(lib, oracle):
    # sizing calls and argument checks need no device (the arithmetic of these two entry points runs on the GPU:
    # tests/test_gpu_parity.py::test_standalone_normalise_and_linear_resample)
    n = C.c_int64()
    assert lib.fa_linear_resample(None, 1000, 3, 48000.0, 16000.0, None, 0, C.byref(n)) == 0 and n.value == 333
    assert lib.fa_linear_resample(None, 1000, 0, 48000.0, 16000.0, None, 0, C.byref(n)) != 0
    z = np.ones((3, 4), np.float32)
    assert lib.fa_mel_normalize_per_feature(z.ctypes.data, 3, 4, 0) == 0 and not z.any()   # no valid frame: all padding
    assert lib.fa_mel_normalize_per_feature(None, 3, 4, 1) != 0
    from fluidaudio_b200.clustering import dendrogram_cut
    rng = np.random.default_rng(5)
    for n in (2, 7, 40):
        xx = oracle.l2_normalize_rows(rng.standard_normal((n, 3)))
        _, z = oracle.centroid_linkage(xx)
        for thr in (0.0, 0.5, 1.0, 2.5, float("nan")):
            assert np.array_equal(dendrogram_cut(z, n, thr), oracle.dendrogram_cut(z, n, thr))


def test_constrained_assignment_host_functions(lib, oracle):
    """The per-chunk Hungarian matching is host code inside the library (exact integer logic, O(chunks K^3)):
    reference KATs (HungarianAssignmentTests.swift, ConstrainedClusterAssignmentTests.swift) and equality with the
    oracle on tie-heavy random problems."""
    from fluidaudio_b200.clustering import ConstrainedClusterAssignment as Cc, HungarianAssignment as H, \
        build_chunk_assignments
    assert H.solve([4, 1, 3, 2, 0, 5, 3, 2, 2], 3) == [1, 0, 2] and H.solve([1, 2, 0, 10], 2) == [1, 0]
    assert H.solve([], 0) == []
    assert H.max_score_assignment([[0.9, 0.1], [0.8, 0.2]]) == [0, 1]
    assert H.max_score_assignment([[0.1, 0.9, 0.3]]) == [1]
    assert H.max_score_assignment([[0.9], [0.5], [0.7]]) == [0, -1, -1]
    assert H.max_score_assignment([[float("nan"), 0.2], [0.6, 0.5]]) == [1, 0]
    assert H.max_score_assignment([]) == [] and H.max_score_assignment([[], []]) == [-1, -1]
    assert Cc.assign([[0.9, 0.3], [0.8, 0.6]], [0, 0]) == [0, 1]
    assert Cc.assign([[0.9, 0.3], [0.8, 0.6]], [0, 1]) == [0, 0]
    assert Cc.assign([[0.9], [0.2]], [0, 0]) == [0, -2]
    assert Cc.assign([[0.1, 0.7, 0.4], [0.5, 0.2, 0.9]], [3, 7]) == [1, 2]
    assert Cc.assign([], []) == [] and Cc.assign([[0.50, 0.55], [0.10, 0.90]], [0, 0]) == [0, 1]
    rng = np.random.default_rng(0)
    for _ in range(300):
        rows, cols = int(rng.integers(1, 5)), int(rng.integers(1, 7))
        sc = np.round(rng.random((rows, cols)), 2)
        if rng.random() < 0.2:
            sc[rng.integers(rows), rng.integers(cols)] = np.inf if rng.random() < 0.5 else np.nan
        assert H.max_score_assignment(sc.tolist()) == oracle.max_score_assignment(sc).tolist()
    n, k = 700, 5
    sc = np.round(rng.random((n, k)), 3)
    chunk = rng.integers(0, 250, n)
    spk = rng.integers(0, 3, n)
    got = np.array(Cc.assign(sc, chunk), np.int32)
    assert np.array_equal(got, oracle.constrained_assign(sc, chunk))
    assert np.array_equal(build_chunk_assignments(chunk, spk, got, 250, 3, k),
                          oracle.build_chunk_assignments(chunk, spk, got, 250, 3, k))
    for c in np.unique(chunk):          # distinct clusters inside a chunk (or -2)
        a = got[chunk == c]
        assert len(set(a[a >= 0].tolist())) == (a >= 0).sum()


# ------------------------------------------------------------------------------------------------ device code on the host
def _compile(src, out):
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-o", out,
                           os.path.join(ROOT, "tests", "emul", src)])
    return C.CDLL(out)


def test_kernel_lane_math_matches_oracle(tmp_path, oracle):
    """mel_core.cuh (the per-lane FFT256 / recombination / banded mel / log the CUDA kernel runs) emulated lane by
    lane on the host vs the oracle: same frames, |delta log-mel| <= 1e-4."""
    L = _compile("mel_emul.cpp", str(tmp_path / "libmel_emul.so"))
    f32p = np.ctypeslib.ndpointer(np.float32, flags="C_CONTIGUOUS")
    L.mel_emul.argtypes = [f32p, C.c_longlong, C.c_float, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_int, f32p,
                           f32p, C.c_float, C.c_int, C.c_longlong, f32p]
    for nm, gen, n in ((80, synth.tone_noise_audio, 16000 * 4 + 137), (128, synth.speech_like_audio, 16000 * 3)):
        a = gen(n)
        ref, T, _ = oracle.mel_flat_transposed(oracle.mel_config(n_mels=nm), a)
        out = np.zeros((T, nm), np.float32)
        assert L.mel_emul(a, a.size, 0.0, 160, 400, 56, 256, np.float32(0.97), nm, oracle.mel_filterbank(512, nm),
                          oracle.hann_window(), np.float32(2.0 ** -24), 0, T, out) == 0
        assert np.abs(out - ref).max() <= 1e-4
    # the float32-pair value type (two frames per warp, FA_MEL_PRECISION_F32) through the same per-lane code: index math of
    # the pair rows, exact-rounded twiddle scalars; float32 transform noise stays inside the bar on these fixtures
    L.mel_emul_f32x2.argtypes = L.mel_emul.argtypes
    for nm, gen, n in ((80, synth.tone_noise_audio, 16000 * 4 + 137), (128, synth.speech_like_audio, 16000 * 3)):
        a = gen(n)
        ref, T, _ = oracle.mel_flat_transposed(oracle.mel_config(n_mels=nm), a)
        out = np.zeros((T, nm), np.float32)
        assert L.mel_emul_f32x2(a, a.size, 0.0, 160, 400, 56, 256, np.float32(0.97), nm, oracle.mel_filterbank(512, nm),
                                oracle.hann_window(), np.float32(2.0 ** -24), 0, T, out) == 0
        assert np.abs(out - ref).max() <= 1e-4
    # legacy compute(): window at offset 0, no padding, no pre-emphasis
    a = synth.tone_noise_audio(8000)
    ref, T = oracle.mel_legacy(oracle.mel_config(n_mels=80), a)
    out = np.zeros((T, 80), np.float32)
    assert L.mel_emul(a, a.size, 0.0, 160, 400, 0, 0, np.float32(0.0), 80, oracle.mel_filterbank(512, 80),
                      oracle.hann_window(), np.float32(2.0 ** -24), 0, T, out) == 0
    assert np.abs(out.T - ref).max() <= 1e-4


def test_merge_control_plane_matches_reference_goldens(tmp_path, golden_dir, oracle):
    """ahc_core.cuh (slot-indexed heap + live bitmap, the code the device master warp runs) driven on the host in the
    merge kernel's order: dendrograms must equal the reference's bit for bit."""
    L = _compile("ahc_emul.cpp", str(tmp_path / "libahc_emul.so"))
    g = np.load(os.path.join(golden_dir, "ahc_reference.npz"))
    for name in sorted({k.rsplit("__", 1)[0] for k in g.files}):
        x = np.ascontiguousarray(g[name + "__x"])
        z = np.zeros((x.shape[0] - 1, 4))
        assert L.ahc_emul(x.ctypes.data_as(C.c_void_p), x.shape[0], x.shape[1], z.ctypes.data_as(C.c_void_p)) == 0
        assert np.array_equal(z, g[name + "__z"]), name
    rng = np.random.default_rng(17)
    for n, d in ((300, 8), (257, 3)):
        x = np.round(rng.standard_normal((n, d)), 1)          # coarse grid: many exactly tied distances
        z = np.zeros((n - 1, 4))
        assert L.ahc_emul(x.ctypes.data_as(C.c_void_p), n, d, z.ctypes.data_as(C.c_void_p)) == 0
        assert np.array_equal(z, oracle.centroid_linkage(x)[1])
    bad = rng.standard_normal((10, 3)); bad[4, 1] = np.nan
    assert L.ahc_emul(bad.ctypes.data_as(C.c_void_p), 10, 3, np.zeros((9, 4)).ctypes.data_as(C.c_void_p)) == 5


# ------------------------------------------------------------------------------------------------ sharding
def test_float32_filter_bound_is_rigorous():
    """The AHC initial pass trusts E_ij = c1 r_i r_j + c2 (n_i + n_j), c1 = 2.02 (D + 3) 2^-24, c2 = 2e-12
    (ahc_kernels.cu: ahc_filter_prep / tile128 / rows) to bracket the reference's sequential double chain from a float32
    inner product of float32-converted inputs, and evaluates the bracket in float32 interval arithmetic.  Restated here in
    numpy (directed rounding through nextafter) and checked on inputs chosen to stress it: unit rows, near-duplicates,
    exact duplicates, rows of very different norm, widths that are not multiples of eight, float32 sums in three orders."""
    rng = np.random.default_rng(7)
    f32, f64 = np.float32, np.float64

    def chain(a, b):                      # fastcluster's sq. distance: sum += (a_k - b_k)^2, every operation rounded
        s = f64(0.0)
        for k in range(a.size):
            d = f64(a[k] - b[k])
            s = f64(s + f64(d * d))
        return s

    def rd(x):                            # float64 -> float32 rounded down / up
        y = f32(x)
        return y if f64(y) <= x else np.nextafter(y, f32(-np.inf))

    def ru(x):
        y = f32(x)
        return y if f64(y) >= x else np.nextafter(y, f32(np.inf))

    worst = 0.0
    for D in (256, 255, 64, 13):
        c1 = 2.02 * (D + 3) * 2.0 ** -24
        c2 = 2e-12
        base = rng.standard_normal((24, D))
        base /= np.linalg.norm(base, axis=1, keepdims=True)
        rows = [base[i] for i in range(24)]
        rows += [base[0] + 1e-7 * rng.standard_normal(D), base[1] * (1 + 1e-9), base[2].copy(), base[3] * 37.5, base[4] * 1e-3,
                 np.round(base[5] * 4) / 4, np.zeros(D)]
        X = np.asarray(rows, f64)
        Xf = X.astype(f32)
        n = (X * X).sum(axis=1)                                   # |x|^2 in double (k ascending in the kernel; any order here)
        r = np.array([ru(np.sqrt(v)) * f32(1.000001) for v in n], f32)
        for i in range(len(rows)):
            for j in range(i):
                exact = chain(X[i], X[j])
                dots = (np.dot(Xf[i], Xf[j]),                                          # library order
                        f32(sum(f32(Xf[i][k] * Xf[j][k]) for k in range(D))),          # sequential, products rounded
                        f32(np.sum((Xf[i][::-1] * Xf[j][::-1]).astype(f32), dtype=f32)))   # reversed
                for dot in dots:
                    dot = f64(dot)
                    approx = (n[i] + n[j]) - 2.0 * dot
                    E = c1 * f64(r[i]) * f64(r[j]) + c2 * (n[i] + n[j])
                    assert approx - E <= exact <= approx + E, (D, i, j)
                    if E > 0:
                        worst = max(worst, abs(approx - exact) / E)
                    # the float32 interval form of the tile kernel's epilogue brackets the same bounds
                    s_lo, s_hi = rd(f64(rd(n[i])) + f64(rd(n[j]))), ru(f64(ru(n[i])) + f64(ru(n[j])))
                    e_up = ru(f64(ru(f64(ru(c1)) * f64(r[i]))) * f64(r[j]) + f64(ru(f64(ru(c2)) * f64(s_hi))))
                    hi = ru(f64(ru(-2.0 * dot + f64(s_hi))) + f64(e_up))
                    lo = rd(f64(rd(-2.0 * dot + f64(s_lo))) - f64(e_up))
                    assert f64(lo) <= approx - E + 1e-300 or f64(lo) <= exact
                    assert f64(lo) <= exact <= f64(hi), (D, i, j)
    assert 0.0 < worst < 0.9, worst     # observed error stays below 90 % of the bound (and the check is not vacuous)


def test_sharding_partitions():
    for count, world in ((512, 8), (64, 8), (10, 4), (3, 8), (0, 2)):
        seen = []
        for r in range(world):
            seen += list(sharding.contiguous_shard(count, r, world))
        assert seen == list(range(count))
        sizes = [len(sharding.contiguous_shard(count, r, world)) for r in range(world)]
        assert max(sizes) - min(sizes) <= 1
    costs = [sharding.ahc_cost(n) for n in (5000, 100, 3000, 3000, 800, 4500, 50, 2000)]
    parts = sharding.lpt_partition(costs, 3)
    assert sorted(sum(parts, [])) == list(range(8))
    loads = [sum(costs[i] for i in p) for p in parts]
    assert max(loads) <= 1.34 * sum(costs) / 3          # LPT bound (4/3 - 1/3m) on the makespan
    assert sharding.lpt_partition(costs, 3) == parts    # deterministic


_WORKER = r"""
import os, sys, numpy as np
sys.path.insert(0, {root!r})
from fluidaudio_b200 import sharding
d = sharding.init_distributed("gloo")
mine = sharding.contiguous_shard(10, d.rank, d.world)
labels = np.array([100 * d.rank + i for i in mine], np.int32)
sharding.barrier(d)
mx = sharding.all_reduce_max(d, 1.5 + d.rank)
sm = sharding.all_reduce_sum(d, len(mine))
got = sharding.gather_labels(d, labels, [len(sharding.contiguous_shard(10, r, d.world)) for r in range(d.world)])
import hashlib
digests = np.stack([np.frombuffer(hashlib.sha256(bytes([i])).digest(), np.uint8) for i in mine])
allh = sharding.gather_bytes(d, digests, [len(sharding.contiguous_shard(10, r, d.world)) for r in range(d.world)])
# the C5 plan: 64 equal meetings over the ranks by LPT, labels come back in partition order
parts = sharding.lpt_partition([sharding.ahc_cost(5000)] * 64, d.world)
mine5 = np.concatenate([np.full(3, m, np.int32) for m in parts[d.rank]])
got5 = sharding.gather_labels(d, mine5, [3 * len(p) for p in parts])
if d.is_root:
    assert mx == 2.5 and sm == 10.0, (mx, sm)
    assert got.tolist() == [0, 1, 2, 3, 4, 105, 106, 107, 108, 109], got.tolist()
    assert allh.shape == (10, 32) and all(allh[i].tobytes() == hashlib.sha256(bytes([i])).digest() for i in range(10))
    assert sorted(sum(parts, [])) == list(range(64)) and all(len(p) == 32 for p in parts)
    assert got5.tolist() == [m for p in parts for m in p for _ in range(3)]
    print("GLOO_OK")
sharding.finalize(d)
"""


def test_two_rank_gloo_plumbing(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(_WORKER.format(root=ROOT))
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT="29533")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                          "--master-addr", "127.0.0.1", "--master-port", "29533", str(script)],
                         env=env, capture_output=True, text=True, timeout=240)
    assert out.returncode == 0, out.stderr[-2000:]
    assert "GLOO_OK" in out.stdout


# ---- embedding-export files (OfflineDiarizerManager.exportEmbeddings, :913-955): host-only code of the library ----
def _random_export(n, seed=0, e=256, r=128):
    from fluidaudio_b200.export_io import EmbeddingExport
    rng = np.random.default_rng(seed)
    return EmbeddingExport(
        chunk_index=np.sort(rng.integers(0, max(1, n // 2), n)).astype(np.int32),
        speaker_index=rng.integers(0, 3, n).astype(np.int32),
        start_frame=rng.integers(0, 500, n).astype(np.int32), end_frame=rng.integers(500, 1000, n).astype(np.int32),
        start_time=rng.random(n) * 1e3, end_time=rng.random(n) * 1e3 + 1e3,
        embedding256=(rng.standard_normal((n, e)) * 10.0 ** rng.integers(-6, 3, (n, e))).astype(np.float32),
        rho128=rng.standard_normal((n, r)) * 10.0 ** rng.integers(-12, 6, (n, r)),
        cluster=rng.integers(-1, 5, n).astype(np.int32))


def test_embedding_export_round_trip_is_bit_exact(lib, tmp_path):
    from fluidaudio_b200.export_io import EmbeddingExport, PreparedDiarization
    for n in (0, 1, 37):
        ex = _random_export(n, seed=n)
        p = tmp_path / f"export_{n}.json"
        ex.write(p)
        back = EmbeddingExport.read(p)
        assert back.count == n
        for f in ("chunk_index", "speaker_index", "start_frame", "end_frame", "cluster"):
            assert np.array_equal(getattr(back, f), getattr(ex, f))
        for f in ("start_time", "end_time", "embedding256", "rho128"):            # bit patterns, not just values
            a, b = getattr(back, f), getattr(ex, f)
            assert a.dtype == b.dtype and a.tobytes() == b.tobytes()
        if n:
            import json                                                              # the file is plain JSON
            doc = json.load(open(p))
            assert len(doc) == n and set(doc[0]) == {"chunkIndex", "speakerIndex", "startFrame", "endFrame", "startTime",
                                                      "endTime", "embedding256", "rho128", "cluster"}
            prep = PreparedDiarization.load(p)
            assert prep.embedding_count == n and prep.segmentation_chunk_count == int(ex.chunk_index.max()) + 1


def test_embedding_export_reads_foundation_style_json(lib, tmp_path):
    """Key order, whitespace, exponents and unknown keys as Foundation's JSONEncoder / other tools may produce."""
    from fluidaudio_b200.export_io import EmbeddingExport
    text = """ [ {"rho128":[1e-05, -3.5E+2 ,0.1], "cluster" : 2, "embedding256":[0.100000001,-7,1.17549435e-38],
                  "endTime":12.5,"startTime":2,"endFrame":40,"startFrame":4,"speakerIndex":1,"chunkIndex":3,
                  "frameWeights":[0.5,{"nested":[1,2,{"x":null}]},"s\\"tr"], "extra": true },
                 {"chunkIndex":4,"speakerIndex":0,"startFrame":5,"endFrame":6,"startTime":0.25,"endTime":0.5,
                  "embedding256":[1,2,3],"rho128":[4,5,6]} ]\n"""
    p = tmp_path / "swift.json"
    p.write_text(text)
    ex = EmbeddingExport.read(p)
    assert ex.count == 2 and ex.embedding256.shape == (2, 3) and ex.rho128.shape == (2, 3)
    assert ex.chunk_index.tolist() == [3, 4] and ex.speaker_index.tolist() == [1, 0]
    assert ex.start_frame.tolist() == [4, 5] and ex.end_frame.tolist() == [40, 6]
    assert ex.start_time.tolist() == [2.0, 0.25] and ex.end_time.tolist() == [12.5, 0.5]
    assert ex.cluster.tolist() == [2, -1]                                           # absent -> -1, as the writer's default
    assert ex.embedding256[0].tolist() == [np.float32(0.1), -7.0, np.float32(1.17549435e-38)]
    assert ex.rho128[0].tolist() == [1e-05, -350.0, 0.1]


def test_embedding_export_errors_are_reported(lib, tmp_path):
    from fluidaudio_b200.export_io import EmbeddingExport
    with pytest.raises(_lib.FluidAudioError) as e:
        EmbeddingExport.read(tmp_path / "missing.json")
    assert e.value.status == 1 and "cannot open" in str(e.value)
    for name, text, what in (("trunc", '[{"chunkIndex":1,"embedding256":[1,2', "expected"),
                             ("ragged", '[{"embedding256":[1,2],"rho128":[1]},{"embedding256":[1],"rho128":[1]}]', "different"),
                             ("notarray", '{"chunkIndex":1}', "expected '['"),
                             ("frac", '[{"chunkIndex":1.5,"embedding256":[],"rho128":[]}]', "integer"),
                             ("tail", '[] x', "trailing")):
        p = tmp_path / f"{name}.json"
        p.write_text(text)
        with pytest.raises(_lib.FluidAudioError) as e:
            EmbeddingExport.read(p)
        assert e.value.status == 1 and what in str(e.value), (name, str(e.value))


def test_same_partition_helper():
    from fluidaudio_b200.export_io import same_partition
    assert same_partition([0, 0, 1, 2, -2], [5, 5, 3, 9, -1])
    assert not same_partition([0, 0, 1], [1, 2, 2])
    assert not same_partition([0, 1], [0, 0])
    assert not same_partition([0, -2], [0, 1])
    assert not same_partition([0, 1], [0, 1, 2])


def test_speaker_constraints_host_function(lib, oracle):
    """fa_speaker_constraints_resolve needs no device; same table as SpeakerCountConstraintsTests.swift."""
    from fluidaudio_b200.clustering import OfflineDiarizerConfig, SpeakerCountConstraints
    cases = [(100, None, None, None), (100, 3, 1, 10), (5, None, 2, 20), (100, None, 10, 5), (100, 0, None, None),
             (100, -5, None, None), (100, None, 0, 5), (100, None, -3, 5), (1, None, None, None), (7, -1, None, None)]
    for n, num, lo, hi in cases:
        got = SpeakerCountConstraints.resolve(n, num, lo, hi)
        assert (got.min_speakers, got.max_speakers) == oracle.speaker_constraints(n, num, lo, hi)
    c = SpeakerCountConstraints.resolve(100, None, 5, 10)
    assert c.needs_adjustment(3) and c.target_count(3) == 5 and c.num_speakers is None    # :104-113
    c = SpeakerCountConstraints.resolve(100, None, 2, 5)
    assert c.needs_adjustment(8) and c.target_count(8) == 5                               # :115-124
    assert not c.needs_adjustment(3) and c.target_count(3) == 3                           # :126-135
    assert SpeakerCountConstraints.resolve(100, 3, 1, 10).num_speakers == 3
    cfg = OfflineDiarizerConfig().with_speakers(min=2, max=4)
    cc = cfg._c_cluster()
    assert (cc.num_speakers, cc.min_speakers, cc.max_speakers) == (_lib.NO_VALUE, 2, 4)
    cc = cfg.with_speakers(exactly=3)._c_cluster()
    assert (cc.num_speakers, cc.min_speakers, cc.max_speakers) == (3, _lib.NO_VALUE, _lib.NO_VALUE)


def test_headers_are_plain_c_and_link(lib, tmp_path):
    """include/*.h compile as C11 with -Wall -Wextra -pedantic -Werror, and a C program linked against the shared
    library runs the host-only part of the ABI (no GPU needed)."""
    exe = tmp_path / "abi_smoke"
    libdir = os.path.dirname(_lib.LIB_PATH)
    subprocess.check_call(["gcc", "-std=c11", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "c", "abi_smoke.c"), "-o", str(exe), "-L", libdir,
                           "-lfluidaudio_b200", f"-Wl,-rpath,{libdir}"])
    out = subprocess.check_output([str(exe)], text=True)
    assert out.startswith("abi ok:")


# ---- timeline reconstruction (OfflineReconstruction.buildSegments): host code of the library vs the oracle -----------
def _synthetic_segmentation(rng, chunks, frames=60, speakers=3, step=20, dur=0.05, k=3):
    """Sliding windows over a piecewise-constant speaker timeline: weights in {~0, ~1}, local slots permuted per chunk."""
    total = step * (chunks - 1) + frames
    truth = np.zeros((total, k), np.float32)
    t = 0
    while t < total:
        length = int(rng.integers(5, 40))
        who = rng.choice(k, size=int(rng.integers(0, 3)), replace=False)
        truth[t:t + length, who] = 1.0
        t += length
    w = np.zeros((chunks, frames, speakers), np.float32)
    hard = np.full((chunks, speakers), -2, np.int32)
    for c in range(chunks):
        perm = rng.permutation(k)[:speakers]
        seg = truth[c * step:c * step + frames]
        for s, cl in enumerate(perm):
            if seg[:, cl].any():
                hard[c, s] = cl
                w[c, :, s] = np.clip(seg[:, cl] * rng.uniform(0.7, 1.0) + rng.uniform(0, 0.05, frames), 0, 1)
    offsets = np.arange(chunks) * step * dur
    return w, hard, offsets, dur, truth


def test_timeline_reconstruction_matches_oracle(lib, oracle):
    from fluidaudio_b200.clustering import OfflineReconstruction
    rng = np.random.default_rng(4)
    for case in range(12):
        chunks = int(rng.integers(1, 30))
        w, hard, offsets, dur, truth = _synthetic_segmentation(rng, chunks)
        kw = dict(min_gap_duration=float(rng.choice([0.0, 0.1, 0.5])), min_segment_duration=float(rng.choice([0.0, 0.2, 1.0])),
                  exclusive_segments=bool(rng.integers(0, 2)))
        use_off = offsets if case % 3 else offsets[: max(1, chunks // 2)]        # missing offsets -> chunk * windowDuration
        got = OfflineReconstruction(dur, window_duration=1.0, **kw).build_segments(w, hard, 3, use_off)
        ref = oracle.build_segments(w, hard, 3, dur, use_off, window_duration=1.0, **kw)
        assert [(s.cluster, s.start_time_seconds, s.end_time_seconds, s.quality_score) for s in got] == \
            [(c, float(a), float(b), float(q)) for c, a, b, q in ref], case
        starts = [s.start_time_seconds for s in got]
        assert starts == sorted(starts) and all(s.speaker_id == f"S{s.cluster + 1}" for s in got)
        if kw["exclusive_segments"]:
            assert all(a.end_time_seconds <= b.start_time_seconds for a, b in zip(got, got[1:]))
        assert all(s.end_time_seconds - s.start_time_seconds >= np.float32(kw["min_segment_duration"]) for s in got)
    # hand-checked cases: two chunks of 4 frames (0.5 s each), one local speaker each, both mapped to cluster 1
    w = np.zeros((2, 4, 2), np.float32)
    w[0, :, 0] = 0.9
    w[1, 2:, 1] = 0.8
    hard = np.array([[1, -2], [-2, 1]], np.int32)
    r = OfflineReconstruction(0.5, window_duration=2.0, min_segment_duration=0.0)
    segs = r.build_segments(w, hard, 2, [0.0, 2.0])
    assert [(s.cluster, s.start_time_seconds, s.end_time_seconds) for s in segs] == [(1, 0.0, 2.0), (1, 3.0, 4.0)]
    assert abs(segs[0].quality_score - 0.9) < 1e-6 and abs(segs[1].quality_score - 0.8) < 1e-6
    merged = OfflineReconstruction(0.5, window_duration=2.0, min_segment_duration=0.0, min_gap_duration=1.0) \
        .build_segments(w, hard, 2, [0.0, 2.0])
    assert [(s.cluster, s.start_time_seconds, s.end_time_seconds) for s in merged] == [(1, 0.0, 4.0)]
    assert abs(merged[0].quality_score - (0.9 * 2 + 0.8 * 1) / 3) < 1e-6          # duration-weighted blend
    assert OfflineReconstruction(0.0).build_segments(w, hard, 2) == []            # frameDuration <= 0 -> []
    assert OfflineReconstruction(0.5).build_segments(np.zeros((0, 0, 0), np.float32), [], 2) == []
    cents = np.random.default_rng(0).standard_normal((2, 7))
    db = OfflineReconstruction.build_speaker_database(merged + segs, cents)      # three segments, all of cluster 1
    odb, ocnt = oracle.build_speaker_database([s.cluster for s in merged + segs], cents)
    assert list(db) == ["S2"] and ocnt.tolist() == [0, 3] and db["S2"].tobytes() == odb[1].tobytes()
    c32 = cents[1].astype(np.float32)
    assert np.array_equal(db["S2"], ((c32 + c32) + c32) * np.float32(1.0 / 3.0))
    none = r.build_segments(w, np.full((2, 2), -2, np.int32), 2, [0.0, 2.0])
    assert all(s.cluster == 0 for s in none)     # zero votes everywhere: the ranking's tie-break picks cluster 0 (:177-186)
