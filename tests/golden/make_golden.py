"""Generates the committed golden fixtures.  Run HERE (the container that has /root/reference):

    python tests/golden/make_golden.py

* ahc_*.npz   inputs + dendrograms produced by the UNMODIFIED reference FastClusterWrapper.cpp
              (oracle/_ref/liboracle_fc.so, built by `make -C oracle ref`) — these pin both the oracle
              restatement (CPU tests) and the CUDA path (GPU tests).
* ahc_large.json  SHA-256 of the reference dendrogram bytes for the BASELINE-size problems (N = 5 000 / 10 000),
              whose inputs are regenerated from seeds (fluidaudio_b200/synth.py) instead of being stored.
* next_rows.npz  the rows either side of the hot path (SURVEY 8f): seeded K-Means runs, UnifiedMelExtractor and LS-EEND
              features from the oracle restatement (`python tests/golden/make_golden.py next` regenerates only these).
* ref_linkage.json  the reference's status and dendrogram SHA-256 for every input on which the tests and smoke() ask for
              its result (oracle.reference_linkage, keyed by a hash of the input bytes), so that those comparisons run
              where the reference cannot be compiled.  Record them by running the whole suite (GPU tests included)
              and smoke() with oracle/_ref built and FA_ORACLE_RECORD_REF=<dir>, then
              `python tests/golden/make_golden.py ref_linkage <dir>`.
* ahc_placements.json  the reference's status and dendrogram SHA-256, and the SHA-256 of the labels cut at 0.6, for the
              linkage problems that reach each placement of the CUDA merge loop and initial pass (PLACEMENT_CASES), plus
              the SHA-256 of the final pipeline labels (oracle.diarize_cluster) of the batch sets (BATCH_SETS).  Inputs
              are regenerated from seeds; recording also checks that the restatement reproduces every dendrogram.
              `python tests/golden/make_golden.py placements` regenerates only this file (several CPU-minutes per
              large case; the cases run in parallel).
* mel_*.npz   log-mel of the reference's own test signal (SortformerStreamingMelTests.swift:17-25 shape) from the
              oracle restatement: the reference has no golden mel values and no Swift toolchain exists here, so
              these pin the oracle against silent drift, not against Apple's vDSP.
"""
import glob
import hashlib
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from fluidaudio_b200 import synth  # noqa: E402
from oracle import oracle as O  # noqa: E402


def ref_linkage(x):
    st, z = O.centroid_linkage(x, use_ref=True)
    assert st == 0
    return z


def next_rows():
    out = {}
    six = np.array([[1.0, 0.0], [1.1, 0.1], [0.0, 1.0], [0.1, 1.1], [-1.0, 0.0], [-0.9, 0.1]])
    for name, (x, k, iters, seed) in {"six_k3_seed42": (six, 3, 100, 42), "six_k3_seed12345": (six, 3, 300, 12345)}.items():
        lab, cen, it = O.kmeans(x, k, iters, seed)
        out[f"kmeans_{name}__labels"], out[f"kmeans_{name}__centroids"] = lab, cen
    emb, _ = synth.speaker_embeddings(300, 64, 5, seed=9)
    lab, cen, best = O.kmeans_ninit(emb.astype(np.float64), 5, 100, 10, 0)
    out["kmeans_ninit_300x64__labels"], out["kmeans_ninit_300x64__centroids"] = lab, cen
    out["kmeans_ninit_300x64__best"] = np.array([best])
    a = synth.tone_noise_audio(16000)
    window = np.concatenate([a[:6000], np.zeros(2000, np.float32)])
    mel, valid = O.unified_mel_features(window, 6000)
    out["unified_8000_valid6000__mel"], out["unified_8000_valid6000__valid"] = mel, np.array([valid])
    cfg = O.lseend_config()
    f1, mean, cnt = O.lseend_features(cfg, a[:4000], np.zeros(23, np.float32), 0)
    f2, mean, cnt = O.lseend_features(cfg, a[4000 - 352:9000], mean, cnt)
    out["lseend__f1"], out["lseend__f2"], out["lseend__mean"], out["lseend__count"] = f1, f2, mean, np.array([cnt])
    np.savez_compressed(os.path.join(HERE, "next_rows.npz"), **out)
    print("next_rows.npz written:", sorted(out))


def pack_ref_linkage(src):
    """Merges the reference records written under `src` into ref_linkage.json, keeping the entries already there."""
    path = os.path.join(HERE, "ref_linkage.json")
    records = json.load(open(path)) if os.path.exists(path) else {}
    for rec in sorted(glob.glob(os.path.join(src, "*.json"))):
        records[os.path.basename(rec)[:-5]] = json.load(open(rec))
    with open(path, "w") as f:
        f.write("{\n" + ",\n".join(f"{json.dumps(k)}: {json.dumps(records[k])}" for k in sorted(records)) + "\n}\n")
    print(f"{len(records)} reference records in {path}")


# ---- linkage placements (tests/test_gpu_cluster_config_space.py) -----------------------------------------------------
# name: (N, D, kind, seed).  kinds: "speaker" = L2-normalised synthetic speaker embeddings (8 speakers); "gauss" = raw
# standard normal rows; "eighths" = standard normal rounded to multiples of 1/8 (exact in binary, so equal distances are
# exact ties); "dupes" = 20 distinct standard normal rows, 200 copies each, shuffled.
PLACEMENT_CASES = {
    "l3_11376x32": (11376, 32, "speaker", 101),
    "l2_11377x32": (11377, 32, "speaker", 102),
    "l2_14176x32": (14176, 32, "speaker", 103),
    "l1_14177x32": (14177, 32, "speaker", 104),
    "l2_ties_12000x8": (12000, 8, "eighths", 105),
    "l1_resident_15000x256": (15000, 256, "speaker", 106),
    "l1_streamed_17000x256": (17000, 256, "speaker", 107),
    "l1_full_18800x64": (18800, 64, "speaker", 108),
    "l1_18808x8": (18808, 8, "speaker", 117),
    "l0_resident_18809x8": (18809, 8, "speaker", 118),
    "l0_streamed_19000x64": (19000, 64, "speaker", 109),
    "l0_tiles_33000x16": (33000, 16, "speaker", 110),
    "tiles_2050x1600": (2050, 1600, "speaker", 111),
    "pad_2048x1": (2048, 1, "gauss", 112),
    "pad_3000x3": (3000, 3, "gauss", 113),
    "pad_2500x300": (2500, 300, "speaker", 114),
    "pad_4097x257": (4097, 257, "speaker", 115),
    "overflow_4000x8": (4000, 8, "dupes", 116),
}
# batches for fa_diarize_cluster_batch: lists of (N, seed) at D = 256; the 17 000-row set is l1_streamed_17000x256's
BATCH_SETS = {
    "four_lanes": [(17000, 107), (400, 201), (400, 202), (400, 203)],
    "two_lanes": [(6000, 204), (6000, 205), (6000, 206)],
}


def placement_input(n, d, kind, seed):
    """(linkage input [n x d] float64, the float32 embeddings it was normalised from or None)."""
    if kind == "speaker":
        emb, _ = synth.speaker_embeddings(n, d, 8, seed=seed)
        return O.l2_normalize_rows(emb.astype(np.float64)), emb
    rng = np.random.default_rng(seed)
    if kind == "gauss":
        return rng.standard_normal((n, d)), None
    if kind == "eighths":
        return np.round(rng.standard_normal((n, d)) * 8.0) / 8.0, None
    assert kind == "dupes" and n % 20 == 0
    return np.repeat(rng.standard_normal((20, d)), n // 20, axis=0)[rng.permutation(n)], None


def batch_set(n, seed):
    """(embeddings float32 [n x 256], rho [n x 128], psi [128]) of one batch set."""
    emb, _ = synth.speaker_embeddings(n, 256, 8, seed=seed)
    rho, psi = synth.synthetic_plda(emb)
    return emb, rho, psi


def _sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def _record_linkage(name):
    n, d, kind, seed = PLACEMENT_CASES[name]
    x, _ = placement_input(n, d, kind, seed)
    st, z = O.centroid_linkage(x, use_ref=True)
    st2, z2 = O.centroid_linkage(x)
    assert st == st2 == 0 and np.array_equal(z, z2), f"{name}: the restatement differs from the reference"
    return name, {"n": n, "d": d, "kind": kind, "seed": seed, "status": st, "z_sha256": _sha(z),
                  "labels_sha256": _sha(O.dendrogram_cut(z, n, 0.6))}


def _record_pipeline(key):
    n, seed = key
    emb, rho, psi = batch_set(n, seed)
    return f"{n}_seed{seed}", {"n": n, "seed": seed,
                               "final_labels_sha256": _sha(O.diarize_cluster(emb, rho, psi, use_ref=True).labels)}


def placements():
    from concurrent.futures import ProcessPoolExecutor
    jobs = sorted({s for sets in BATCH_SETS.values() for s in sets}, key=lambda s: -s[0])
    names = sorted(PLACEMENT_CASES, key=lambda k: -PLACEMENT_CASES[k][0] * PLACEMENT_CASES[k][1] ** 0.5)
    with ProcessPoolExecutor(os.cpu_count()) as pool:
        pipes = [pool.submit(_record_pipeline, k) for k in jobs]
        links = [pool.submit(_record_linkage, k) for k in names]
        out = {"linkage": dict(f.result() for f in links), "pipelines": dict(f.result() for f in pipes)}
    with open(os.path.join(HERE, "ahc_placements.json"), "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
        f.write("\n")
    print(f"ahc_placements.json written: {len(out['linkage'])} linkages, {len(out['pipelines'])} pipelines")


def main():
    O.build()
    if len(sys.argv) > 1 and sys.argv[1] == "next":
        return next_rows()
    if len(sys.argv) > 1 and sys.argv[1] == "placements":
        assert O.ref_available(), "oracle/_ref/liboracle_fc.so missing: run `make -C oracle ref` where the reference exists"
        return placements()
    if len(sys.argv) > 2 and sys.argv[1] == "ref_linkage":
        return pack_ref_linkage(sys.argv[2])
    assert O.ref_available(), "oracle/_ref/liboracle_fc.so missing: run `make -C oracle ref` where /root/reference exists"
    rng = np.random.default_rng(2024)
    cases = {}
    # BASELINE config 1: 100 x 256, 4 speakers
    emb, _ = synth.speaker_embeddings(100, 256, 4, weights=(0.4, 0.3, 0.2, 0.1), seed=1)
    cases["c1_100x256"] = O.l2_normalize_rows(emb.astype(np.float64))
    cases["random_64x7"] = rng.standard_normal((64, 7))
    base = rng.standard_normal((20, 5))
    cases["duplicates_80x5"] = np.repeat(base, 4, axis=0)[rng.permutation(80)]
    cases["lattice_64x3"] = np.array([[i, j, k] for i in range(4) for j in range(4) for k in range(4)], float)
    cases["two_points"] = np.array([[1.0, 0.0], [0.0, 1.0]])
    cases["line_9x1"] = np.array([[0.0], [1.0], [2.5], [2.6], [7.0], [7.05], [7.1], [20.0], [21.0]])
    out = {}
    for name, x in cases.items():
        x = np.ascontiguousarray(x, np.float64)
        out[name + "__x"] = x
        out[name + "__z"] = ref_linkage(x)
    np.savez_compressed(os.path.join(HERE, "ahc_reference.npz"), **out)

    large = {}
    for name, (n, k, w, seed) in {"c5_5000x256_seed0": (5000, 4, (0.4, 0.3, 0.2, 0.1), 0),
                                  "c3_10000x256_seed42": (10000, 8, None, 42)}.items():
        emb, _ = synth.speaker_embeddings(n, 256, k, weights=w, seed=seed)
        x = O.l2_normalize_rows(emb.astype(np.float64))
        z = ref_linkage(x)
        labels = O.dendrogram_cut(z, n, 0.6)
        rho, psi = synth.synthetic_plda(emb)
        pipe = O.diarize_cluster(emb, rho, psi, use_ref=True)
        large[name] = {"n": n, "speakers": k, "weights": w, "seed": seed,
                       "final_labels_sha256": hashlib.sha256(pipe.labels.tobytes()).hexdigest(),
                       "final_centroids": int(pipe.centroids.shape[0]), "vbx_iterations": int(len(pipe.vbx.elbos)),
                       "vbx_last_elbo": float(pipe.vbx.elbos[-1]),
                       "z_sha256": hashlib.sha256(z.tobytes()).hexdigest(),
                       "labels_sha256": hashlib.sha256(labels.tobytes()).hexdigest(),
                       "clusters": int(labels.max() + 1), "last_merge_distance": float(z[-1, 2])}
        print(name, large[name])
    with open(os.path.join(HERE, "ahc_large.json"), "w") as f:
        json.dump(large, f, indent=1)

    mel = {}
    a = synth.tone_noise_audio(16000 * 2 + 137)
    mel["audio"] = a
    for nm in (80, 128):
        m, ml, nf = O.mel_flat_transposed(O.mel_config(n_mels=nm), a)
        mel[f"center_{nm}"] = m
    m, ml = O.mel_legacy(O.mel_config(n_mels=128), a)
    mel["legacy_128"] = m
    m, ml, nf = O.mel_flat_transposed(O.mel_config(n_mels=80, preemph=0.0, log_floor=1e-10, log_floor_mode=1,
                                                   window_periodic=True), a, padding_mode=1)
    mel["lseend_prepadded_80"] = m
    mel["hann_400"] = O.hann_window(400, False)
    mel["filterbank_80"] = O.mel_filterbank(512, 80)
    np.savez_compressed(os.path.join(HERE, "mel_oracle.npz"), **mel)
    next_rows()
    print("golden fixtures written to", HERE)


if __name__ == "__main__":
    main()
