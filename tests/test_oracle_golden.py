"""CPU tests that PIN THE ORACLE (oracle/ is test infrastructure; see its headers).

1. against the unmodified reference C++ (oracle/_ref/liboracle_fc.so where it was built, else its results recorded for
   the same inputs, tests/golden/ref_linkage.json) and against golden dendrograms that reference produced
   (tests/golden/ahc_reference.npz);
2. against an independent implementation (scipy centroid linkage; numpy float64 mel pipeline);
3. against the reference's own unit tests, ported as known-answer tests:
   Tests/FluidAudioTests/Diarizer/Offline/AHCClusteringTests.swift, ASR/Parakeet/Streaming/
   AudioMelSpectrogramTests.swift, EouChunkSizeFrameCountTests.swift, Diarizer/Offline/VDSPOperationsTests.swift.
"""
import hashlib
import json
import os

import numpy as np
import pytest

from fluidaudio_b200 import synth


# ------------------------------------------------------------------------------------------------ AHC: pinning
def test_restatement_reproduces_reference_goldens_bit_exact(oracle, golden_dir):
    g = np.load(os.path.join(golden_dir, "ahc_reference.npz"))
    names = sorted({k.rsplit("__", 1)[0] for k in g.files})
    assert len(names) >= 6
    for name in names:
        x, z_ref = g[name + "__x"], g[name + "__z"]
        st, z = oracle.centroid_linkage(x)
        assert st == 0
        assert np.array_equal(z, z_ref), f"{name}: restatement differs from the reference dendrogram"


def test_restatement_equals_compiled_reference_on_fresh_inputs(oracle):
    rng = np.random.default_rng(7)
    for n, d in ((2, 3), (3, 1), (17, 4), (200, 16), (600, 256)):
        x = rng.standard_normal((n, d))
        st1, z1 = oracle.centroid_linkage(x)
        st2, z2 = oracle.centroid_linkage(x, use_ref=True)
        assert st1 == st2 == 0 and np.array_equal(z1, z2)
    x = np.repeat(rng.standard_normal((30, 6)), 5, axis=0)[rng.permutation(150)]   # exact ties
    assert np.array_equal(oracle.centroid_linkage(x)[1], oracle.centroid_linkage(x, use_ref=True)[1])


def test_large_reference_hashes_match_restatement(oracle, golden_dir):
    meta = json.load(open(os.path.join(golden_dir, "ahc_large.json")))
    m = meta["c5_5000x256_seed0"]
    emb, _ = synth.speaker_embeddings(m["n"], 256, m["speakers"], weights=m["weights"], seed=m["seed"])
    x = oracle.l2_normalize_rows(emb.astype(np.float64))
    st, z = oracle.centroid_linkage(x)
    assert st == 0
    assert hashlib.sha256(z.tobytes()).hexdigest() == m["z_sha256"]
    labels = oracle.dendrogram_cut(z, m["n"], 0.6)
    assert hashlib.sha256(labels.tobytes()).hexdigest() == m["labels_sha256"]
    assert labels.max() + 1 == m["clusters"]


def test_status_codes_match_reference_contract(oracle):
    import ctypes as C
    L = oracle.lib()
    x = np.ones((3, 2))
    z = np.zeros(8)
    assert L.oracle_centroid_linkage(None, 3, 2, z.ctypes.data, 8) == 1
    assert L.oracle_centroid_linkage(x.ctypes.data, 0, 2, z.ctypes.data, 8) == 0
    assert L.oracle_centroid_linkage(x.ctypes.data, 3, 0, z.ctypes.data, 8) == 1
    assert L.oracle_centroid_linkage(x.ctypes.data, 3, 2, z.ctypes.data, 7) == 3
    assert L.oracle_centroid_linkage(x.ctypes.data, 1, 2, z.ctypes.data, 0) == 0
    assert L.oracle_centroid_linkage(x.ctypes.data, 2 ** 31, 2, z.ctypes.data, 8) == 2
    bad = np.array([[0.0, 1.0], [np.nan, 0.0], [1.0, 1.0]])
    assert oracle.centroid_linkage(bad)[0] == 5
    assert oracle.centroid_linkage(bad, use_ref=True)[0] == 5


def test_restatement_agrees_with_scipy_centroid_linkage(oracle):
    from scipy.cluster.hierarchy import linkage
    rng = np.random.default_rng(3)
    x = rng.standard_normal((300, 12))
    st, z = oracle.centroid_linkage(x)
    zs = linkage(x, method="centroid")
    assert np.array_equal(z[:, :2], zs[:, :2]) and np.array_equal(z[:, 3], zs[:, 3])
    assert np.abs(z[:, 2] - zs[:, 2]).max() < 1e-12


# ------------------------------------------------------------------------------------------------ AHC: reference KATs
def test_ahc_empty_single_and_zero_dim(oracle):
    for use_ref in (False, True):
        assert oracle.ahc_cluster(np.zeros((0, 3)), 0.7, use_ref).size == 0
        assert oracle.ahc_cluster(np.array([[1.0, 0, 0]]), 0.7, use_ref).tolist() == [0]
        assert oracle.ahc_cluster(np.zeros((3, 0)), 0.7, use_ref).tolist() == [0, 0, 0]


def test_ahc_reference_unit_tests(oracle):
    for use_ref in (False, True):
        same = oracle.ahc_cluster(np.tile([1.0, 2.0, 3.0], (5, 1)), 0.7, use_ref)
        assert len(set(same.tolist())) == 1
        g1 = [[1.0, 0, 0], [0.9, 0.1, 0], [0.95, 0.05, 0]]
        g2 = [[0, 1.0, 0], [0, 0.9, 0.1], [0, 0.95, 0.05]]
        r = oracle.ahc_cluster(np.array(g1 + g2), 0.8, use_ref)
        assert len(set(r[:3].tolist())) == 1 and len(set(r[3:].tolist())) == 1 and r[0] != r[3]
        four = np.array([[1.0, 0, 0], [0.9, 0.1, 0], [0, 1.0, 0], [0, 0.9, 0.1]])
        assert len(set(oracle.ahc_cluster(four, 0.5, use_ref).tolist())) == 2
        assert len(set(oracle.ahc_cluster(four, 1.5, use_ref).tolist())) == 1
        eye = np.eye(3)
        ids = sorted(set(oracle.ahc_cluster(eye, 0.5, use_ref).tolist()))
        assert ids == list(range(len(ids)))
        assert len(set(oracle.ahc_cluster(eye, 2.0, use_ref).tolist())) == 1
        assert len(set(oracle.ahc_cluster(eye, 0.0, use_ref).tolist())) == 3


def test_cut_is_the_swift_traversal_not_scipy_fcluster(oracle):
    """Centroid linkage has inversions; the Swift cut uses each node's own distance (SURVEY §0 D8)."""
    def py_cut(z, n, thr):
        thr = 0.0 if np.isnan(thr) else max(0.0, min(2.0, thr))
        left = {n + m: int(z[m, 0]) for m in range(n - 1)}
        right = {n + m: int(z[m, 1]) for m in range(n - 1)}
        dist = {n + m: z[m, 2] for m in range(n - 1)}
        lab, nxt, stack = [-1] * n, 0, [2 * n - 2]
        while stack:
            node = stack.pop()
            if node < n:
                if lab[node] == -1:
                    lab[node] = nxt; nxt += 1
                continue
            if dist[node] <= thr:
                q = [node]
                while q:
                    c = q.pop()
                    if c < n: lab[c] = nxt
                    else: q += [left[c], right[c]]
                nxt += 1
            else:
                stack += [left[node], right[node]]
        remap, out = {}, []
        for v in lab:
            remap.setdefault(v, len(remap)); out.append(remap[v])
        return np.array(out, np.int32)
    rng = np.random.default_rng(11)
    inversions = 0
    for trial in range(40):
        n = int(rng.integers(5, 60))
        x = oracle.l2_normalize_rows(rng.standard_normal((n, 3)))
        _, z = oracle.centroid_linkage(x)
        inversions += int((np.diff(z[:, 2]) < 0).any())
        for thr in (0.0, 0.3, 0.8, 1.2, 2.0, 5.0, -1.0, float("nan")):
            assert np.array_equal(oracle.dendrogram_cut(z, n, thr), py_cut(z, n, thr))
    assert inversions > 0


def test_l2_normalize_matches_reference_vdsp_test(oracle):
    # VDSPOperationsTests.swift: l2Normalize([3,4]) == [0.6, 0.8]; zero rows stay zero (AHCClustering.swift:88)
    out = oracle.l2_normalize_rows(np.array([[3.0, 4.0], [0.0, 0.0]]))
    assert np.allclose(out[0], [0.6, 0.8], atol=1e-15) and np.all(out[1] == 0)


# ------------------------------------------------------------------------------------------------ VBx / assignment
def _numpy_vbx(x, psi, init, S, Fa=0.07, Fb=0.8, iters=20, eps=1e-4):
    T, D = x.shape
    g = np.zeros((T, S)); g[np.arange(T), init] = 1
    g = np.exp(7 * g - (7 * g).max(1, keepdims=True)); g /= g.sum(1, keepdims=True); g /= g.sum(1, keepdims=True)
    pi = np.full(S, 1 / S)
    phi = np.maximum(psi, 1e-12)
    rho = x * np.sqrt(phi)
    G = -0.5 * ((x ** 2).sum(1) + D * np.log(2 * np.pi))
    prev, elbos = -np.inf, []
    for it in range(iters):
        invL = 1 / np.maximum(1 + (Fa / Fb) * g.sum(0)[:, None] * phi[None], 1e-12)
        alpha = (Fa / Fb) * invL * (g.T @ rho)
        phiT = ((alpha ** 2 + invL) * phi).sum(1)
        logp = Fa * (rho @ alpha.T - 0.5 * phiT + G[:, None]) + np.log(np.maximum(pi, 1e-8))
        mx = logp.max(1, keepdims=True)
        e = np.exp(logp - mx); s = e.sum(1, keepdims=True)
        g = e / s
        ll = (mx + np.log(s)).sum()
        pi = g.sum(0) / g.sum()
        elbo = ll + Fb * 0.5 * (np.log(invL).sum() - invL.sum() - (alpha ** 2).sum() + invL.size)
        elbos.append(elbo)
        if it > 0 and abs(elbo - prev) < eps:
            break
        prev = elbo
    return g, pi, np.array(elbos)


def test_vbx_matches_independent_numpy_restatement(oracle):
    emb, who = synth.speaker_embeddings(600, 256, 5, seed=5)
    rho, psi = synth.synthetic_plda(emb)
    init = oracle.ahc_cluster(emb.astype(np.float64), 0.6)
    S = len(set(init.tolist()))
    out = oracle.vbx_refine(rho, psi, init)
    g, pi, elbos = _numpy_vbx(rho, psi, init, S)
    assert out.num_clusters == S and len(out.elbos) == len(elbos)
    assert np.abs(out.gamma - g).max() < 1e-9 and np.abs(out.pi - pi).max() < 1e-10
    assert np.abs((out.elbos - elbos) / elbos).max() < 1e-12
    assert np.allclose(out.gamma.sum(1), 1.0, atol=1e-12)
    assert np.all(np.diff(out.elbos) > -1e-6)          # EM never decreases the bound
    assert np.array_equal(out.hard, g.argmax(1))


def test_pipeline_recovers_speakers_and_filters_nan(oracle):
    emb, who = synth.speaker_embeddings(400, 256, 4, weights=(0.4, 0.3, 0.2, 0.1), seed=9)
    emb[7, 100] = np.inf
    emb[123, 0] = np.nan
    rho, psi = synth.synthetic_plda(np.nan_to_num(emb, posinf=0.0))
    r = oracle.diarize_cluster(emb, rho, psi)
    assert r.training_indices.size == 398 and 7 not in r.training_indices
    ok = np.isfinite(emb).all(1)
    # AHC separates the four speakers exactly; VBx (with the synthetic PLDA and only 400 frames) may then merge
    # some of them — every true speaker must still land in exactly one final cluster
    init_pairs = set(zip(who[r.training_indices].tolist(), r.initial.tolist()))
    assert len(init_pairs) == 4
    pairs = set(zip(who[ok].tolist(), r.labels[ok].tolist()))
    assert len(pairs) == 4
    K = r.centroids.shape[0]
    assert r.labels.shape == (400,) and 1 <= K <= 4 and r.labels.max() < K and r.centroids.shape[1] == 256


def test_assign_first_maximum_wins(oracle):
    cents = np.array([[1.0, 0.0], [2.0, 0.0], [0.0, 1.0]])     # centroids 0 and 1 are collinear: equal cosine
    emb = np.array([[3.0, 0.0], [0.0, 5.0], [0.0, 0.0]])
    labels, scores = oracle.assign_embeddings(emb, cents, want_scores=True)
    assert labels.tolist() == [0, 2, 0]
    assert scores[0, 0] == scores[0, 1] == 1.0


# ------------------------------------------------------------------------------------------------ mel
def test_mel_goldens_are_reproduced(oracle, golden_dir):
    g = np.load(os.path.join(golden_dir, "mel_oracle.npz"))
    a = g["audio"]
    for nm in (80, 128):
        m, ml, nf = oracle.mel_flat_transposed(oracle.mel_config(n_mels=nm), a)
        assert np.array_equal(m, g[f"center_{nm}"])
    assert np.array_equal(oracle.mel_legacy(oracle.mel_config(n_mels=128), a)[0], g["legacy_128"])
    assert np.array_equal(oracle.hann_window(400, False), g["hann_400"])
    assert np.array_equal(oracle.mel_filterbank(512, 80), g["filterbank_80"])


def test_mel_matches_independent_float64_numpy_pipeline(oracle):
    a = synth.tone_noise_audio(16000 + 137)
    for nm in (80, 128):
        w = oracle.hann_window().astype(np.float64)
        fb = oracle.mel_filterbank(512, nm).astype(np.float64)
        p = np.zeros(a.size + 512)
        p[256] = a[0]
        p[257:257 + a.size - 1] = a[1:].astype(np.float64) - float(np.float32(0.97)) * a[:-1].astype(np.float64)
        T = 1 + (a.size + 512 - 400) // 160
        fr = np.zeros((T, 512))
        for f in range(T):
            s = f * 160 + 56
            av = min(400, p.size - s)
            fr[f, 56:56 + av] = p[s:s + av] * w[:av]
        ref = np.log(np.abs(np.fft.rfft(fr, axis=1)) ** 2 @ fb.T + float(np.float32(2.0 ** -24)))
        m64, ml, _ = oracle.mel_flat_transposed(oracle.mel_config(n_mels=nm, precision=1), a)
        assert ml == T and np.abs(m64 - ref).max() < 5e-6
        m32, _, _ = oracle.mel_flat_transposed(oracle.mel_config(n_mels=nm), a)       # THE oracle
        m32b, _, _ = oracle.mel_flat_transposed(oracle.mel_config(n_mels=nm, precision=2), a)   # float32 FFT variant
        assert np.abs(m32 - ref).max() < 5e-5
        assert np.abs(m32b - m32).max() < 1e-4


def test_mel_reference_structure_tests(oracle):
    """AudioMelSpectrogramTests.swift + EouChunkSizeFrameCountTests.swift."""
    cfg = oracle.mel_config()
    m, ml = oracle.mel_legacy(cfg, np.zeros(16000, np.float32))
    assert ml == 98 and m.shape == (128, 98) and (m < 0).all()
    assert oracle.mel_legacy(cfg, np.full(800, 0.1, np.float32))[1] > 0
    flat, ml, nf = oracle.mel_flat(cfg, np.zeros(16000, np.float32))
    assert nf > 0 and flat.size == 128 * nf
    w = oracle.hann_window()
    assert w.size == 400 and np.allclose(w, w[::-1], atol=1e-6) and abs(w[0]) < 1e-6 and abs(w[-1]) < 1e-6
    assert abs(w[200] - 1.0) < 0.01
    fb = oracle.mel_filterbank()
    assert fb.shape == (128, 257) and (fb >= 0).all()
    # StreamingChunkSize: chunkSamples = (melFrames - 1) * hop for 17 / 64(?) / 129 frames; formula check instead
    for n in (1000, 2000, 5000, 8000, 10080, 12000, 15000, 20000, 25000, 30000, 2560, 20480):
        assert oracle.mel_flat(cfg, np.full(n, 0.1, np.float32))[1] == 1 + (n + 512 - 400) // 160
    assert oracle.mel_frame_count(cfg, 2560) == 17 and oracle.mel_frame_count(cfg, 20480) == 129


def test_mel_modes_and_guards(oracle):
    cfg = oracle.mel_config(n_mels=80, pad_to=16)
    a = synth.tone_noise_audio(5000)
    m, ml, nf = oracle.mel_flat_transposed(cfg, a)
    assert ml == 32 and nf == 32 and m.shape == (32, 80)
    m, ml, nf = oracle.mel_flat_transposed(cfg, a[:4000])
    assert ml == 26 and nf == 32 and np.all(m[26:] == 0)              # padded rows are zero
    # prePadded: (n - nFFT)/hop + 1 with truncating division; below 352 samples -> no frame
    assert oracle.mel_frame_count(cfg, 400, 1) == 1 and oracle.mel_frame_count(cfg, 352, 1) == 0
    out, ml, nf = oracle.mel_flat_transposed(cfg, np.zeros(0, np.float32))
    assert ml == 0 and nf == 1 and out.size == 80 and np.all(out == 0)
    # expectedFrameCount beyond the signal: all-zero frames -> log(floor)
    m, ml, nf = oracle.mel_flat_transposed(oracle.mel_config(n_mels=80), a[:800], expected_frames=12)
    assert ml == 12 and np.allclose(m[11], np.log(np.float32(2.0 ** -24)), atol=1e-6)
    # streamed pre-padded == batch centre (SortformerStreamingMelTests.swift:84-132), within 1e-5
    full, T, _ = oracle.mel_flat_transposed(oracle.mel_config(n_mels=128), a)
    padded = np.concatenate([np.zeros(256, np.float32), a, np.zeros(256, np.float32)])
    # pre-emphasis must see the true previous sample, so apply the same filter by passing preemph through the pad
    pre, T2, _ = oracle.mel_flat_transposed(oracle.mel_config(n_mels=128), padded, padding_mode=1)
    assert T2 == T
    assert np.abs(pre[2:-2] - full[2:-2]).max() < 1e-5


def test_adapters(oracle):
    x = np.arange(24, dtype=np.float32).reshape(6, 4) ** 1.5
    y = oracle.normalize_per_feature(x, 4)
    assert np.all(y[4:] == 0) and np.allclose(y[:4].mean(0), 0, atol=1e-6)
    assert np.allclose(y[:4].std(0, ddof=1), 1.0, atol=1e-3)
    assert np.all(oracle.normalize_per_feature(x, 0) == 0)
    planar = np.stack([np.arange(10, dtype=np.float32), np.arange(10, dtype=np.float32) * 3,
                       np.zeros(10, np.float32)])
    mono = planar.mean(0)
    assert np.allclose(oracle.linear_resample(planar, 16000, 16000), mono)
    half = oracle.linear_resample(planar, 32000, 16000)
    assert half.size == 5 and np.allclose(half, mono[::2])
    up = oracle.linear_resample(planar, 8000, 16000)
    assert up.size == 20 and np.allclose(up[:19], np.interp(np.arange(19) / 2, np.arange(10), mono), atol=1e-5)


# ------------------------------------------------------------------------------------------------ constrained assignment
def test_hungarian_and_constrained_assignment_reference_kats(oracle):
    """HungarianAssignmentTests.swift + ConstrainedClusterAssignmentTests.swift, exact integer outputs."""
    assert oracle.hungarian_solve(np.array([[4, 1, 3], [2, 0, 5], [3, 2, 2]])).tolist() == [1, 0, 2]
    assert oracle.hungarian_solve(np.array([[1, 2], [0, 10]])).tolist() == [1, 0]
    assert oracle.hungarian_solve(np.zeros((0, 0))).size == 0
    assert oracle.max_score_assignment([[0.9, 0.1], [0.8, 0.2]]).tolist() == [0, 1]
    assert oracle.max_score_assignment([[0.1, 0.9, 0.3]]).tolist() == [1]
    assert oracle.max_score_assignment([[0.9], [0.5], [0.7]]).tolist() == [0, -1, -1]
    assert oracle.max_score_assignment([[np.nan, 0.2], [0.6, 0.5]]).tolist() == [1, 0]
    assert oracle.max_score_assignment(np.zeros((2, 0))).tolist() == [-1, -1]
    assert oracle.constrained_assign([[0.9, 0.3], [0.8, 0.6]], [0, 0]).tolist() == [0, 1]
    assert oracle.constrained_assign([[0.9, 0.3], [0.8, 0.6]], [0, 1]).tolist() == [0, 0]
    assert oracle.constrained_assign([[0.9], [0.2]], [0, 0]).tolist() == [0, -2]
    assert oracle.constrained_assign([[0.1, 0.7, 0.4], [0.5, 0.2, 0.9]], [3, 7]).tolist() == [1, 2]
    assert oracle.constrained_assign([[0.50, 0.55], [0.10, 0.90]], [0, 0]).tolist() == [0, 1]
    assert oracle.constrained_assign(np.zeros((0, 2)), []).size == 0
    # optimality against brute force on small random problems
    import itertools
    rng = np.random.default_rng(1)
    for _ in range(200):
        n = int(rng.integers(1, 6))
        cost = rng.integers(0, 20, (n, n))
        best = min(sum(cost[i, p[i]] for i in range(n)) for p in itertools.permutations(range(n)))
        a = oracle.hungarian_solve(cost)
        assert sorted(a.tolist()) == list(range(n)) and sum(cost[i, a[i]] for i in range(n)) == best


def test_adapter_restatements_against_numpy(oracle):
    """UnifiedMelExtractor per-feature normalisation and LS-EEND cumulative mean normalisation (SURVEY 8f rank 3):
    the C restatements against straightforward numpy float64 formulas."""
    from fluidaudio_b200 import synth
    a = synth.tone_noise_audio(16000 * 4)
    window = np.concatenate([a[:40000], np.zeros(24000, np.float32)])
    mel, valid = oracle.unified_mel_features(window, 40000)
    total = window.size // 160 + 1
    assert mel.shape == (128, total) and valid == 40000 // 160
    raw, _, _ = oracle.mel_flat_transposed(oracle.mel_config(n_mels=128), window, 0.0, 0, expected_frames=total)
    x = raw[:valid].astype(np.float64)
    ref = (x - x.mean(axis=0)) / (x.std(axis=0, ddof=1) + 1e-5)
    assert np.abs(mel[:, :valid].T - ref).max() < 2e-4
    assert not mel[:, valid:].any()
    m0, v0 = oracle.unified_mel_features(window, 100)                  # fewer samples than one hop: everything zero
    assert v0 == 0 and not m0.any()

    cfg = oracle.lseend_config()
    f1, mean1, c1 = oracle.lseend_features(cfg, a[:16000], np.zeros(23, np.float32), 0)
    f2, mean2, c2 = oracle.lseend_features(cfg, a[16000 - 352:40000], mean1, c1)
    assert c1 == f1.shape[0] == (16000 - 512) // 160 + 1 and c2 == c1 + f2.shape[0]
    raw1, ml1, _ = oracle.mel_flat_transposed(cfg, a[:16000], 0.0, 1, None)
    raw2, ml2, _ = oracle.mel_flat_transposed(cfg, a[16000 - 352:40000], 0.0, 1, None)
    y = np.concatenate([raw1[:ml1], raw2[:ml2]]).astype(np.float64) / np.log(10.0)
    cum = np.cumsum(y, axis=0) / np.arange(1, y.shape[0] + 1)[:, None]
    got = np.concatenate([f1, f2])
    assert np.abs(got - (y - cum)).max() < 1e-4
    assert np.abs(mean2 - cum[-1]).max() < 1e-4
    assert not got[0].any()                                            # first frame minus its own mean


# ---- K-Means re-clustering + speaker-count constraints (SURVEY 8f rank 4) ---------------------------------------------
class _SwiftLCG:
    """KMeansClustering.SeededRNG (:212-223) + the Swift stdlib's next(upperBound:) / Double.random(in: a...b),
    restated independently of the oracle to generate the reference test's inputs."""
    def __init__(self, seed):
        self.state = seed & (2 ** 64 - 1)

    def next(self):
        self.state = (self.state * 6364136223846793005 + 1442695040888963407) & (2 ** 64 - 1)
        return self.state

    def next_below(self, upper):
        m = self.next() * upper
        if (m & (2 ** 64 - 1)) < upper:
            t = (2 ** 64 - upper) % upper
            while (m & (2 ** 64 - 1)) < t:
                m = self.next() * upper
        return m >> 64

    def double_closed(self, lo, hi):
        rand = self.next_below((1 << 53) + 1)
        if rand == (1 << 53):
            return hi
        return (hi - lo) * (rand * 2.0 ** -53) + lo


def test_kmeans_reference_tests(oracle):
    """Tests/FluidAudioTests/Diarizer/Clustering/KMeansClusteringTests.swift, case by case."""
    six = np.array([[1.0, 0.0], [1.1, 0.1], [0.0, 1.0], [0.1, 1.1], [-1.0, 0.0], [-0.9, 0.1]])
    lab, cen, _ = oracle.kmeans(six, 3, 100, 42)                                     # :10-31
    assert lab.size == 6 and len(set(lab.tolist())) == 3
    lab, _, _ = oracle.kmeans(np.array([[1.0, 0.0], [1.1, 0.1], [0.9, 0.2]]), 1, 100, 42)   # :33-49
    assert lab.tolist() == [0, 0, 0]
    lab, cen, _ = oracle.kmeans(np.array([[1.0, 0.0], [0.0, 1.0]]), 5, 100, 42)      # :51-67
    assert lab.tolist() == [0, 1] and np.array_equal(cen, [[1.0, 0.0], [0.0, 1.0]])
    lab, cen, _ = oracle.kmeans(np.array([[1.0, 0.0], [1.0, 0.0], [0.0, 1.0], [0.0, 1.0]]), 2, 100, 42)   # :69-86
    assert cen.shape[0] == 2 and lab.size == 4
    a = oracle.kmeans(six, 3, 300, 12345)[0]                                         # :90-109
    assert np.array_equal(a, oracle.kmeans(six, 3, 300, 12345)[0])
    rng = _SwiftLCG(42)                                                              # :113-131
    emb = np.array([[rng.double_closed(-1.0, 1.0) for _ in range(192)] for _ in range(20)])
    lab, _, _ = oracle.kmeans(emb, 3, 100, 42)
    assert lab.size == 20 and len(set(lab.tolist())) == 3


def test_kmeans_restatement_properties(oracle):
    from fluidaudio_b200 import synth
    emb, who = synth.speaker_embeddings(500, 64, 5, seed=9)
    x = emb.astype(np.float64)
    lab, cen, it = oracle.kmeans(x, 5, 100, 3)
    xn = x / np.linalg.norm(x, axis=1, keepdims=True)
    d = ((xn[:, None, :] - cen[None]) ** 2).sum(-1)
    assert np.array_equal(lab, d.argmin(1))                                          # fixed point of the assignment step
    for j in range(5):                                                               # centroids = means of their members
        if (lab == j).any():
            assert np.abs(cen[j] - xn[lab == j].mean(0)).max() < 1e-12
    best_lab, best_cen, best = oracle.kmeans_ninit(x, 5, 100, 10, 0)
    inertias = []
    for s in range(10):
        l, c, _ = oracle.kmeans(x, 5, 100, s)
        inertias.append(((xn - c[l]) ** 2).sum())
    assert best == int(np.argmin(inertias)) and np.array_equal(best_lab, oracle.kmeans(x, 5, 100, best)[0])
    # an empty cluster is re-seeded from a data point: duplicates force it
    dup = np.repeat(np.eye(3), 4, axis=0)
    l, c, _ = oracle.kmeans(dup, 3, 50, 1)
    assert len(set(l.tolist())) == 3


def test_speaker_constraints_reference_tests(oracle):
    """Tests/FluidAudioTests/Diarizer/Offline/SpeakerCountConstraintsTests.swift (resolve; -> (min, max))."""
    r = oracle.speaker_constraints
    assert r(100) == (1, 100)                            # :10-20
    assert r(100, 3, 1, 10) == (3, 3)                    # :22-32
    assert r(5, None, 2, 20) == (2, 5)                   # :34-43
    assert r(100, None, 10, 5) == (5, 5)                 # :47-56
    assert r(100, 0) == (1, 1) and r(100, -5) == (1, 1)  # :60-80
    assert r(100, None, 0, 5)[0] == 1 and r(100, None, -3, 5)[0] == 1   # :82-100


def test_next_row_goldens(oracle, golden_dir):
    """The committed fixtures of the 8f rows (K-Means, UnifiedMelExtractor, LS-EEND) are reproduced bit for bit."""
    import os
    from fluidaudio_b200 import synth
    g = np.load(os.path.join(golden_dir, "next_rows.npz"))
    six = np.array([[1.0, 0.0], [1.1, 0.1], [0.0, 1.0], [0.1, 1.1], [-1.0, 0.0], [-0.9, 0.1]])
    for name, (k, iters, seed) in {"six_k3_seed42": (3, 100, 42), "six_k3_seed12345": (3, 300, 12345)}.items():
        lab, cen, _ = oracle.kmeans(six, k, iters, seed)
        assert np.array_equal(lab, g[f"kmeans_{name}__labels"]) and cen.tobytes() == g[f"kmeans_{name}__centroids"].tobytes()
    emb, _ = synth.speaker_embeddings(300, 64, 5, seed=9)
    lab, cen, best = oracle.kmeans_ninit(emb.astype(np.float64), 5, 100, 10, 0)
    assert best == int(g["kmeans_ninit_300x64__best"][0]) and np.array_equal(lab, g["kmeans_ninit_300x64__labels"])
    assert cen.tobytes() == g["kmeans_ninit_300x64__centroids"].tobytes()
    a = synth.tone_noise_audio(16000)
    mel, valid = oracle.unified_mel_features(np.concatenate([a[:6000], np.zeros(2000, np.float32)]), 6000)
    assert valid == int(g["unified_8000_valid6000__valid"][0]) and mel.tobytes() == g["unified_8000_valid6000__mel"].tobytes()
    cfg = oracle.lseend_config()
    f1, mean, cnt = oracle.lseend_features(cfg, a[:4000], np.zeros(23, np.float32), 0)
    f2, mean, cnt = oracle.lseend_features(cfg, a[4000 - 352:9000], mean, cnt)
    assert f1.tobytes() == g["lseend__f1"].tobytes() and f2.tobytes() == g["lseend__f2"].tobytes()
    assert mean.tobytes() == g["lseend__mean"].tobytes() and cnt == int(g["lseend__count"][0])


def test_kmeans_against_independent_python_restatement(oracle):
    """A second, independent restatement of KMeansClustering.clusterWithCentroids (:39-92) in plain Python floats —
    seeded shuffle, first-k picks, strict-< assignment, index-order sums, empty-cluster re-seeding — must give the C++
    oracle's labels and centroids bit for bit."""
    def py_kmeans(emb, k, iters, seed):
        n, d = len(emb), len(emb[0])
        k = min(k, n)
        if n <= k:
            return list(range(n)), [list(map(float, e)) for e in emb]
        rng = _SwiftLCG(seed)
        x = []
        for e in emb:
            s = 0.0
            for v in e:
                s += v * v
            norm = s ** 0.5
            x.append([v * (1.0 / norm) for v in e] if norm > 1e-10 else list(e))
        idx = list(range(n))
        amount, cur = n, 0
        while amount > 1:
            r = rng.next_below(amount)
            amount -= 1
            idx[cur], idx[cur + r] = idx[cur + r], idx[cur]
            cur += 1
        cen = [list(x[i]) for i in idx[:k]]
        assign = [0] * n
        for _ in range(iters):
            fresh = []
            for p in x:
                best, bd = 0, float("inf")
                for j, c in enumerate(cen):
                    dist = 0.0
                    for a, b in zip(p, c):
                        t = a - b
                        dist += t * t
                    if dist < bd:
                        best, bd = j, dist
                fresh.append(best)
            if fresh == assign:
                break
            assign = fresh
            sums = [[0.0] * d for _ in range(k)]
            counts = [0] * k
            for p, a in zip(x, assign):
                counts[a] += 1
                for q in range(d):
                    sums[a][q] += p[q]
            cen = []
            for j in range(k):
                if counts[j] > 0:
                    inv = 1.0 / counts[j]
                    cen.append([v * inv for v in sums[j]])
                else:
                    cen.append(list(x[rng.next_below(n)]))
        return assign, cen

    rng = np.random.default_rng(8)
    for n, d, k, seed in ((12, 3, 3, 0), (40, 8, 5, 7), (25, 4, 6, 42), (9, 2, 9, 1), (30, 5, 4, 12345)):
        emb = rng.standard_normal((n, d)) + 3.0 * rng.integers(0, 3, (n, 1))
        if n == 25:
            emb[5:15] = emb[5]                     # duplicates: provokes an empty cluster and its re-seeding
        lab, cen, _ = oracle.kmeans(emb, k, 50, seed)
        plab, pcen = py_kmeans(emb.tolist(), k, 50, seed)
        assert lab.tolist() == plab
        assert np.array(pcen, np.float64).tobytes() == cen.tobytes()


# ------------------------------------------------------------------------------------------------ AudioConverter stage
def test_resampler_spec_and_reference_length_contract(oracle):
    """The documented Kaiser-sinc filter (the library's stand-in for the closed AVAudioConverter: PARITY UNPINNED for
    values) restated in float64: unit pass band, > 110 dB stop band, output length = Int(n / ratio) within 1 % of the
    nominal count (AudioConverterTests.swift:129-176), mixdown = float32 mean in channel order (:401-409)."""
    for rate, dur, expect in ((44100, 1.0, 16000), (48000, 0.5, 8000), (8000, 2.0, 32000)):
        n = int(rate * dur)
        assert abs(oracle.resample_output_count(n, rate, 16000) - expect) <= 0.01 * expect
    assert oracle.resample_output_count(1000, 16000, 16000) == 1000
    t = np.arange(48000) / 48000.0
    for f0, lo, hi in ((1000.0, 0.9999, 1.0001), (6000.0, 0.999, 1.001), (9000.0, 0.0, 3e-6), (20000.0, 0.0, 3e-6)):
        y = oracle.sinc_resample(np.sin(2 * np.pi * f0 * t).astype(np.float32), 48000, 16000)[2000:-2000].astype(np.float64)
        assert y.size == 16000 - 4000 and lo <= np.sqrt(2 * np.mean(y * y)) <= hi, f0
    x = np.random.default_rng(1).standard_normal(4000).astype(np.float32)
    assert np.array_equal(oracle.sinc_resample(x, 16000, 16000), x)
    L, M, half, fc = oracle.sinc_design(44100, 16000)
    assert (L, M, half) == (160, 441, 67) and abs(fc - 0.94 * 160 / 441) < 1e-15
    # constant in -> the same constant out (rows are normalised to unit DC gain), away from the edges
    y = oracle.sinc_resample(np.full(5000, 0.25, np.float32), 44100, 16000)
    assert np.abs(y[100:-100] - 0.25).max() < 1e-7
    st = np.array([[1.0, 2.0, 3.0], [3.0, 2.0, -3.0]], np.float32)
    assert np.array_equal(oracle.mixdown(st), np.array([2.0, 2.0, 0.0], np.float32))
    i16 = np.array([[16384, -32768]], np.int16)
    assert np.array_equal(oracle.mixdown(i16), np.array([0.5, -1.0], np.float32))
    # one channel through linearResample's arithmetic equals the mono lerp
    m = np.linspace(-1, 1, 1000, dtype=np.float32)
    lin = oracle.linear_resample(np.stack([m, m, m]), 48000, 16000)
    assert lin.size == 333 and np.abs(lin - m[::3][:333]).max() < 1e-6


def test_timed_cpu_arm_matches_the_oracle(oracle):
    """oracle_mel_fast.cpp — the float32-FFT, SIMD-across-frames CPU implementation bench.py times as the reference arm —
    agrees with the parity oracle within the spread of two float32 FFTs (2e-4), frame counts exact."""
    for nm, n, last in ((80, 16000 * 20 + 77, 0.0), (128, 16000 * 7, 0.25), (80, 401, 0.0), (80, 5, -0.5)):
        a = synth.tone_noise_audio(n, seed=nm)
        cfg = oracle.mel_config(n_mels=nm)
        got, ml = oracle.mel_fast_flat_transposed(cfg, a, last)
        ref, rml, _ = oracle.mel_flat_transposed(cfg, a, last=last)
        assert ml == rml and got.shape == ref.shape and np.abs(got - ref).max() <= 2e-4


def test_oracle_against_a_nemo_style_torch_stft_featurizer(oracle):
    """The one external claim the reference makes about its mel values: NemotronMelExtractor matches NeMo's PyTorch
    log-mel to max |delta| ~ 9e-3 (Documentation/Benchmarks.md:149).  NeMo's AudioToMelSpectrogramPreprocessor is
    pre-emphasis 0.97 -> torch.stft(n_fft 512, hop 160, win 400, symmetric Hann, centred) -> |.|^2 -> librosa Slaney
    filterbank (norm='slaney', htk=False) -> log(x + 2^-24).  Rebuilt here from torch.stft (float32, zero padding like the
    Swift code) and an independent float64 restatement of librosa.filters.mel: the oracle must sit well inside the
    reference's own tolerance, and its float32 filterbank within float32 rounding of librosa's formula."""
    torch = pytest.importorskip("torch")

    def hz_to_mel(f):
        f = np.asarray(f, float)
        return np.where(f >= 1000.0, 15.0 + np.log(np.maximum(f, 1e-10) / 1000.0) / (np.log(6.4) / 27.0), f / (200.0 / 3))

    def mel_to_hz(m):
        m = np.asarray(m, float)
        return np.where(m >= 15.0, 1000.0 * np.exp((np.log(6.4) / 27.0) * (m - 15.0)), (200.0 / 3) * m)

    def librosa_slaney(n_mels):
        fftfreqs = np.linspace(0, 8000, 257)
        mel_f = mel_to_hz(np.linspace(hz_to_mel(0.0), hz_to_mel(8000.0), n_mels + 2))
        fdiff, ramps = np.diff(mel_f), mel_f[:, None] - fftfreqs[None, :]
        w = np.stack([np.maximum(0, np.minimum(-ramps[i] / fdiff[i], ramps[i + 2] / fdiff[i + 1])) for i in range(n_mels)])
        return w * (2.0 / (mel_f[2:n_mels + 2] - mel_f[:n_mels]))[:, None]

    for gen, seconds in ((synth.tone_noise_audio, 4), (synth.speech_like_audio, 3)):
        a = gen(16000 * seconds)
        x = torch.from_numpy(a)
        y = torch.cat([x[:1], x[1:] - 0.97 * x[:-1]])
        spec = torch.stft(y, 512, 160, 400, window=torch.hann_window(400, periodic=False), center=True, pad_mode="constant",
                          return_complex=True)
        power = (spec.real ** 2 + spec.imag ** 2).numpy().astype(np.float64)
        for nm in (80, 128):
            fb = librosa_slaney(nm)
            assert np.abs(fb - oracle.mel_filterbank(512, nm)).max() <= 5e-7
            nemo = np.log(fb @ power + 2.0 ** -24).T
            ref, T, _ = oracle.mel_flat_transposed(oracle.mel_config(n_mels=nm), a)
            assert nemo.shape == ref.shape
            assert np.abs(nemo - ref).max() <= 1e-3            # measured 5e-5 .. 1.5e-4; the reference documents 9e-3
