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


def main():
    O.build()
    if len(sys.argv) > 1 and sys.argv[1] == "next":
        return next_rows()
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
