"""The clustering phase across the kernels and placements its host code chooses between, against the reference and the
float64 oracle.

* AHC linkage: every master level (3, 2, 1 with 16-bit heap indices and part of the master state in global memory, 0),
  resident and streamed node vectors, every CTA full, and each initial nearest-neighbour pass (exact, float32 filter with
  the per-row or the tiled pass 2, filter abandoned for the exact pass) are reached by choosing N and D alone, with no
  FA_AHC_FORCE_* hook.  fa_ahc_last_placement tells each case which path it ran; the expected placements are those of
  a 148-SM B200 (147 worker CTAs).  Dendrograms are compared by SHA-256 with the compiled reference's
  (tests/golden/ahc_placements.json, recorded by `python tests/golden/make_golden.py placements`).
* Batch lanes: a set too large for resident placement streamed on 36 workers beside three small sets, and three sets
  sharing the SMs two at a time, each equal to its single-set run and to the reference pipeline.
* VBx on each of its four paths (two-kernel with and without the rho tile, four-kernel with alpha in shared memory or
  read through L2) at the edges of the speaker count S and of the 128-frame blocks, and on every configuration axis;
  centroids on both paths; cosine assignment bit-identical, scores included; K-Means bit-identical.

Known divergence, not tested: for D above about 7 196 the merge kernel's shared-memory target vector does not fit and
the linkage returns FA_RUNTIME_ERROR where the reference succeeds.

Run with -s to see the placement of every linkage and the largest deviation per path.
"""
import ctypes as C
import hashlib
import importlib.util
import json
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from fluidaudio_b200 import _lib, synth
from fluidaudio_b200 import clustering as cl

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_spec = importlib.util.spec_from_file_location("make_golden", os.path.join(ROOT, "tests", "golden", "make_golden.py"))
MG = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(MG)
GOLD = json.load(open(os.path.join(ROOT, "tests", "golden", "ahc_placements.json")))

# (master level, resident, worker CTAs, slots per CTA, initial pass) on 148 SMs; initial pass: 0 exact, 1 filter + rows
# kernel, 2 filter + ahc_filter_tile_kernel<true>, 3 filter abandoned for the exact pass
EXPECTED = {
    "l3_11376x32": (3, 1, 89, 128, 1),
    "l2_11377x32": (2, 1, 89, 128, 1),
    "l2_14176x32": (2, 1, 111, 128, 1),
    "l1_14177x32": (1, 1, 111, 128, 1),
    "l2_ties_12000x8": (2, 1, 94, 128, 1),
    "l1_resident_15000x256": (1, 1, 138, 109, 1),
    "l1_streamed_17000x256": (1, 0, 133, 0, 1),
    "l1_full_18800x64": (1, 1, 147, 128, 1),       # 147 x 128 slots: every CTA full
    "l1_18808x8": (1, 1, 147, 128, 1),
    "l0_resident_18809x8": (0, 1, 147, 128, 1),
    "l0_streamed_19000x64": (0, 0, 147, 0, 1),
    "l0_tiles_33000x16": (0, 0, 147, 0, 2),        # no per-tile minimum buffer (N x N/64 floats > 64 MB)
    "tiles_2050x1600": (3, 1, 147, 14, 2),         # D > 1 536: the rows kernel's x_i does not fit 48 KB
    "pad_2048x1": (3, 1, 16, 128, 1),              # D mod 8 != 0: zero-padded GEMM k dimension
    "pad_3000x3": (3, 1, 24, 125, 1),
    "pad_2500x300": (3, 1, 28, 90, 1),
    "pad_4097x257": (3, 1, 38, 108, 1),
    # 20 distinct rows x 200 copies: 20 x 200 x 199 / 2 = 398 000 exact-duplicate pairs below the diagonal, more than
    # the 64 N = 256 000 candidates the list holds
    "overflow_4000x8": (3, 1, 32, 125, 3),
}
REACHED = set()
MAXDEV = {}


def _note(path, dev):
    MAXDEV[path] = max(MAXDEV.get(path, 0.0), float(dev))


def _sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def last_placement():
    out = np.zeros(6, np.int32)
    _lib.load().fa_ahc_last_placement(out.ctypes.data)
    return tuple(int(v) for v in out)


# ================================================================================================ AHC linkage
def test_case_table_matches_the_golden_file():
    assert set(EXPECTED) == set(MG.PLACEMENT_CASES) == set(GOLD["linkage"])
    for name, (n, d, kind, seed) in MG.PLACEMENT_CASES.items():
        rec = GOLD["linkage"][name]
        assert (rec["n"], rec["d"], rec["kind"], rec["seed"], rec["status"]) == (n, d, kind, seed, 0), name


@pytest.mark.parametrize("name", sorted(MG.PLACEMENT_CASES))
def test_linkage_placement_is_bit_exact(gpu_lib, oracle, name):
    n, d, kind, seed = MG.PLACEMENT_CASES[name]
    rec = GOLD["linkage"][name]
    x, emb = MG.placement_input(n, d, kind, seed)
    st, z = cl.centroid_linkage(x)
    got = last_placement()
    print(f"\n  {name}: placement (level, resident, workers, slots, initial pass, SMs) = {got}", end="")
    assert got[5] == 148, f"the expected placements are those of a 148-SM B200, this device has {got[5]} SMs"
    assert got[:5] == EXPECTED[name], (name, got)
    REACHED.add(got[:5])
    assert st == 0 and _sha(z) == rec["z_sha256"], name
    labels = cl.dendrogram_cut(z, n, 0.6)
    assert _sha(labels) == rec["labels_sha256"], name
    if emb is not None:   # AHCClustering.cluster normalises the raw embeddings to the same x
        assert np.array_equal(cl.AHCClustering().cluster(emb.astype(np.float64), 0.6), labels), name
        assert last_placement() == got


# ================================================================================================ batch lanes
@pytest.mark.parametrize("batch", sorted(MG.BATCH_SETS))
def test_batch_lanes_equal_single_runs_and_reference(gpu_lib, oracle, batch):
    """four_lanes: the 17 000-row set cannot be resident, so four lanes of 36 workers run and it is streamed beside the
    three small sets; two_lanes: 6 000 x 256 needs 56 resident workers, so the three sets share the SMs two at a time."""
    sets = [MG.batch_set(n, seed) for n, seed in MG.BATCH_SETS[batch]]
    psi = sets[0][2]
    assert all(np.array_equal(s[2], psi) for s in sets)
    emb = np.concatenate([s[0] for s in sets])
    rho = np.concatenate([s[1] for s in sets])
    offs = np.concatenate([[0], np.cumsum([s[0].shape[0] for s in sets])]).astype(np.int64)
    labels, infos = cl.OfflineClusterer(psi=psi).cluster_batch(emb, rho, offs)
    for m, ((n, seed), (e, r, _)) in enumerate(zip(MG.BATCH_SETS[batch], sets)):
        part = labels[offs[m]:offs[m + 1]]
        single = cl.OfflineClusterer(psi=psi).cluster(e, r)
        assert np.array_equal(part, single.labels), (batch, m)
        assert _sha(part) == GOLD["pipelines"][f"{n}_seed{seed}"]["final_labels_sha256"], (batch, m)
        assert infos[m]["training_count"] == n


# ================================================================================================ VBx
def vbx_path(S, D):
    """The path refine_device takes (vbx_kernels.cu: fused_path, use_tile, alpha_smem)."""
    fused = 8 * (S * D + 2 * S + 128 * S + 128)
    if S <= 64 and fused <= 200 * 1024:
        return "two-kernel, rho tile" if fused + 8 * D * 129 <= 200 * 1024 else "two-kernel, no tile"
    return "four-kernel, alpha in smem" if 8 * (S * D + 2 * S + 128) <= 200 * 1024 else "four-kernel, alpha via L2"


def vbx_case(T, S, D, seed):
    emb, _ = synth.speaker_embeddings(T, max(256, D), 6, seed=seed)
    rho, psi = synth.synthetic_plda(emb, D)
    rng = np.random.default_rng(seed)
    m = min(S, T)   # S is passed explicitly, so fewer frames than speakers is allowed
    init = rng.permutation(np.concatenate([np.arange(m), rng.integers(0, S, T - m)])).astype(np.int32)
    return rho, psi, init


def gpu_vbx(rho, psi, init, S, max_it, eps, smoothing):
    T, D = rho.shape
    cfg = _lib.VbxConfig(0.07, 0.8, max_it, eps, smoothing)
    cap = max(max_it, 1)
    gamma, pi, elbos = np.zeros((T, S)), np.zeros(S), np.zeros(cap)
    hard, its = np.zeros(T, np.int32), C.c_int32()
    _lib.check(_lib.load().fa_vbx_refine(rho.ctypes.data, T, D, psi.ctypes.data, psi.size, _lib.ptr(init), S,
                                         C.byref(cfg), gamma.ctypes.data, pi.ctypes.data, elbos.ctypes.data,
                                         hard.ctypes.data, C.byref(its)), "fa_vbx_refine")
    return gamma, pi, elbos[:its.value].copy(), hard


def oracle_vbx(oracle, rho, psi, init, S, max_it, eps, smoothing):
    """oracle.vbx_refine with S given (it also runs without initial labels, where the wrapper would infer S = 1)."""
    T, D = rho.shape
    gamma, pi, elbos = np.zeros((T, S)), np.zeros(S), np.zeros(max(max_it, 1))
    hard = np.zeros(T, np.int32)
    cfg = oracle.VbxConfig(0.07, 0.8, max_it, eps, smoothing)
    its = oracle.lib().oracle_vbx_refine(rho, T, D, psi, psi.size, _lib.ptr(init), C.byref(cfg), S, gamma, pi, elbos,
                                         hard)
    return gamma, pi, elbos[:its].copy(), hard


# (T, S, D, seed, max_iterations, epsilon, init_smoothing, with initial labels)
_DEF = (20, 1e-4, 7.0, True)
VBX_CASES = []
for _S in (1, 8, 9, 34, 35, 63, 64, 65, 195, 196, 1024, 1025):                      # S edges of every path at D = 128
    VBX_CASES.append((_S + 1000 if _S > 256 else 1000, _S, 128, 300 + _S) + _DEF)
    VBX_CASES.append((_S, _S, 128, 400 + _S) + _DEF)                                # one frame per speaker
for _S in (9, 35, 65, 196):                                                         # frame-block edges on every path
    for _T in (129, 8193, 16385) + ((77,) if _S < 77 else ()):
        VBX_CASES.append((_T, _S, 128, 500 + _T + _S) + _DEF)
for _S in (48, 49, 63, 64):                                                         # D = 400: S <= 64 off the fused path
    VBX_CASES.append((1000, _S, 400, 600 + _S) + _DEF)
VBX_CASES.append((8193, 49, 400, 700) + _DEF)
for _S in (8, 65):                                                                  # configuration axes, both path kinds
    for _cfg in ((0, 1e-4, 7.0, True), (1, 1e-4, 7.0, True), (2, 1e-4, 7.0, True), (20, 0.0, 7.0, True),
                 (20, 1e-4, -1.0, True), (20, 1e-4, 7.0, False), (20, 1e-4, -1.0, False)):
        VBX_CASES.append((1000, _S, 128, 800 + _S) + _cfg)


def _run_vbx_cases(oracle, cases):
    """GPU runs in order; the oracle runs in threads (its ctypes calls release the GIL)."""
    inputs = [vbx_case(T, S, D, seed) for T, S, D, seed, *_ in cases]

    def ora(i):
        T, S, D, seed, max_it, eps, sm, labelled = cases[i]
        rho, psi, init = inputs[i]
        return oracle_vbx(oracle, rho, psi, init if labelled else None, S, max_it, eps, sm)

    with ThreadPoolExecutor(max(2, min(16, os.cpu_count() or 2))) as pool:
        futures = [pool.submit(ora, i) for i in range(len(cases))]
        for i, (T, S, D, seed, max_it, eps, sm, labelled) in enumerate(cases):
            rho, psi, init = inputs[i]
            g = gpu_vbx(rho, psi, init if labelled else None, S, max_it, eps, sm)
            yield cases[i], inputs[i], g, futures[i].result()


def test_vbx_paths_match_the_oracle(gpu_lib, oracle):
    for case, (rho, psi, init), (g, p, e, h), (og, op, oe, oh) in _run_vbx_cases(oracle, VBX_CASES):
        T, S, D, seed, max_it, eps, sm, labelled = case
        path = vbx_path(S, D)
        # a convergence decision that rounding could flip is a borderline input, not a finding: change its seed
        assert eps == 0 or not np.any(np.abs(np.abs(np.diff(oe)) - eps) < 1e-6), f"borderline input {case}: new seed"
        assert e.size == oe.size, (case, e.size, oe.size)
        assert np.array_equal(h, oh), case
        fused = path.startswith("two-kernel")
        dg, dp = np.abs(g - og).max(), np.abs(p - op).max()
        de = np.abs((e - oe) / oe).max() if oe.size else 0.0
        _note(f"VBx {path}: gamma", dg)
        _note(f"VBx {path}: pi", dp)
        _note(f"VBx {path}: ELBO (relative)", de)
        assert dg <= (1e-9 if fused else 1e-8), (case, dg)
        assert dp <= (1e-9 if fused else 1e-10), (case, dp)
        assert de <= (1e-10 if fused else 1e-9), (case, de)


# ================================================================================================ centroids
@pytest.mark.parametrize("S", [9, 65])
def test_centroids_both_paths_match_the_oracle(gpu_lib, oracle, S):
    """S <= 64: centroid_acc16_kernel + fold; S > 64: accumulate + finish.  gamma and pi come from GPU VBx runs."""
    cases = [(T, S, 128, 900 + T + S) + _DEF for T in (1000, 8193)]
    for (T, *_), (rho, psi, init), (g, p, e, h), _ in _run_vbx_cases(oracle, cases):
        assert not np.any(np.abs(p / 1e-7 - 1.0) <= 1e-6), "a pi at the 1e-7 activity threshold: choose another seed"
        out = cl.VBxOutput(g, p, h, S, e)
        rng = np.random.default_rng(T + S)
        for E in (1, 255, 256, 257):
            emb = rng.standard_normal((T, E))
            cents = cl.compute_centroids(emb, out)
            ocents = oracle.compute_centroids(emb, oracle.VBxOutput(g, p, h, S, e), init)
            assert cents.shape == ocents.shape, (T, S, E)
            dev = np.abs(cents - ocents).max() if cents.size else 0.0
            _note(f"centroids S {'<=' if S <= 64 else '>'} 64", dev)
            assert dev <= (1e-12 if S <= 64 else 1e-9), (T, S, E, dev)


# ================================================================================================ assignment
def _same_bits(a, b):
    na, nb = np.isnan(a), np.isnan(b)
    return np.array_equal(na, nb) and np.array_equal(a[~na].view(np.int64), b[~nb].view(np.int64))


@pytest.mark.parametrize("K", [1, 7, 8, 9, 16, 17, 64])
def test_assignment_is_bit_identical(gpu_lib, oracle, K):
    """assign_tiled_kernel: 8-centroid groups x 32-wide dimension tiles x 128-row CTAs, with rows whose squared norm
    underflows (1e-170), overflows (1e200), is zero or non-finite, a zero centroid and a duplicated one (first maximum
    wins)."""
    rng = np.random.default_rng(K)
    for E in (1, 31, 32, 33, 255, 257):
        for N in (256, 257, 255):
            cen = rng.standard_normal((K, E))
            if K >= 2:
                cen[1] = 0.0
            if K >= 3:
                cen[K - 1] = cen[0]
            emb = rng.standard_normal((N, E))
            emb[0] *= 1e-170
            emb[1] *= 1e200
            emb[2] = 0.0
            emb[3, E // 2] = np.nan
            emb[4, 0] = np.inf
            emb[5, E - 1] = -np.inf
            emb[6:12] = cen[0] * rng.uniform(0.5, 2.0, (6, 1))   # their maximum is at centroid 0 and its duplicate
            labels, scores = cl.assign_embeddings(emb, cen, want_scores=True)
            olabels, oscores = oracle.assign_embeddings(emb, cen, want_scores=True)
            assert np.array_equal(labels, olabels), (K, E, N)
            assert _same_bits(scores, oscores), (K, E, N)
            fin = np.isfinite(oscores)
            _note("assignment scores", np.abs(scores[fin] - oscores[fin]).max() if fin.any() else 0.0)


# ================================================================================================ K-Means
def test_kmeans_is_bit_identical(gpu_lib, oracle):
    rng = np.random.default_rng(31)
    for k in (1, 9, 64, 1024):
        for n in (k + 1, 4 * k):
            for d in (1, 33):
                emb = rng.standard_normal((n, d))
                lab, cen = cl.KMeansClustering.cluster_with_centroids(emb, k, 300, 17)
                ol, oc, _ = oracle.kmeans(emb, k, 300, 17)
                assert np.array_equal(lab, ol) and cen.tobytes() == oc.tobytes(), (k, n, d)
    emb = rng.standard_normal((300, 33))
    lab, cen, best = cl.KMeansClustering.cluster_with_centroids_n_init(emb, 9, 100, 10, 3)
    ol, oc, ob = oracle.kmeans_ninit(emb, 9, 100, 10, 3)
    assert best == ob and np.array_equal(lab, ol) and cen.tobytes() == oc.tobytes()
    # three distinct points and five clusters: the seeding picks duplicates, so clusters run empty and are re-seeded
    dup = np.repeat(rng.standard_normal((3, 33)), 10, axis=0)
    for seed in (1, 2, 3):
        lab, cen = cl.KMeansClustering.cluster_with_centroids(dup, 5, 50, seed)
        ol, oc, _ = oracle.kmeans(dup, 5, 50, seed)
        assert np.array_equal(lab, ol) and cen.tobytes() == oc.tobytes(), seed
    # more than 1 024 clusters is refused, not approximated
    emb = rng.standard_normal((2000, 4))
    labels, cents, rows, best = np.zeros(2000, np.int32), np.zeros((1025, 4)), C.c_int32(), C.c_int32()
    st = _lib.load().fa_kmeans_cluster(emb.ctypes.data, 2000, 4, 1025, 10, 1, 0, labels.ctypes.data, cents.ctypes.data,
                                       1025, C.byref(rows), C.byref(best))
    assert st == 8  # FA_STATUS_UNSUPPORTED


# ================================================================================================ summary
def test_every_placement_was_reached_and_report():
    """Last in the file: every placement of the linkage table ran (and matched the reference) in this session."""
    missing = set(EXPECTED.values()) - REACHED
    print("\n  largest |deviation| from the oracle per path:")
    for path in sorted(MAXDEV):
        print(f"    {path:45s} {MAXDEV[path]:.3g}")
    assert not missing, f"placements not reached: {sorted(missing)}"
