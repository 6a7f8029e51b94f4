"""The heat maps and features that oracle/pin_against_reference.py feeds the reference, rebuilt from seeds.

They are functions of the seeded generators of synth.py (and of the edge-case frames below), so the fixtures under
tests/golden/ store only the small inputs and the reference's outputs; tests/conftest.py puts these arrays back
under the names the fixtures had.  Every builder consumes its random streams in the order the pinning did."""
from __future__ import annotations

import importlib

import numpy as np


def _synth():
    return importlib.import_module("vatl4pose-wacv2024_b200.synth")


def edge_maps():
    """(E,17,64,48) fp32 frames built to hit the edge cases of SURVEY.md §8a."""
    rng = np.random.default_rng(99)
    base = rng.normal(0, 0.02, (17, 64, 48)).astype(np.float32)
    frames = []
    f = base.copy()                                   # 0: plateaus {1,1}, 0.5 and 0.49
    f[0] = 0; f[0, 10, 10] = 1; f[0, 10, 11] = 1; f[0, 30, 30] = .5; f[0, 40, 20] = .49
    f[1] = -np.abs(f[1]) - 0.1                        # all-negative joint: no peak survives
    f[2] = np.minimum(f[2], 0); f[2, 5, 5] = 0        # max == 0
    f[3] = 0; f[3, 0, 0] = 2; f[3, 63, 47] = 2        # ties -> first index; corners (no 1/4 px)
    f[4] = 0; f[4, 1, 1] = 1; f[4, 1, 2] = .5         # px==1: not strictly interior
    f[5] = 0; f[5, 2, 2] = 1; f[5, 2, 3] = .5; f[5, 3, 2] = .7; f[5, 1, 2] = .7   # dy sign 0
    f[6] = 0; f[6, 62, 46] = 1; f[6, 61, 46] = .2     # px==46,py==62: not interior
    f[7] = 0; f[7, 61, 45] = 1; f[7, 61, 44] = .2; f[7, 60, 45] = .3              # last interior
    f[8] = 0.25                                       # constant positive: interior is all plateau
    f[9] = 0; f[9, 0, 10] = -1                        # zeros everywhere but one negative
    f[10] = 0; f[10, 20, :] = 1                       # a full ridge row
    f[11] = 0; f[11, 31, 23] = 3; f[11, 31, 24] = 3; f[11, 32, 23] = 3            # plateau argmax
    frames.append(f)
    g = -np.abs(base) - 1.0                           # 1: every joint negative -> NaN peak mean
    frames.append(g.astype(np.float32))
    z = np.zeros_like(base)                           # 2: all-zero frame
    frames.append(z)
    frames.append(base.copy())                        # 3: pure noise
    return np.stack(frames).astype(np.float32)


def scan_inputs():
    """scan.npz: ten track frames, then the edge-case frames.  Returns H, is_prev, is_next, boxes."""
    synth = _synth()
    rng = np.random.default_rng(0)
    n = 10
    ids, ip, inx = synth.track_flags(n, rng, mean_len=4.0)
    H = synth.heatmaps(n, seed=0, track_ids=ids)
    E = edge_maps()
    H = np.concatenate([H, E], axis=0)
    ne = E.shape[0]
    ip = np.r_[ip, np.array([0, 1, 1, 0][:ne], np.uint8)]
    inx = np.r_[inx, np.array([1, 1, 0, 0][:ne], np.uint8)]
    return H, ip, inx, synth.boxes_xyxy(H.shape[0], seed=0)


def next_inputs():
    """next.npz heat maps: 14 frames in which, inside a track, most joints stay put and a few move by whole pixels
    (TPC discriminative).  Returns H, is_prev, is_next, boxes and the generator, which the pinning goes on using."""
    synth = _synth()
    rng = np.random.default_rng(21)
    n = 14
    ids, ip, inx = synth.track_flags(n, rng, mean_len=5.0)
    H = synth.heatmaps(n, seed=21, track_ids=ids)
    for i in range(1, n):
        if ip[i]:
            H[i] = H[i - 1] + rng.normal(0, 1e-4, H[i].shape).astype(np.float32)
            for j in rng.choice(17, size=int(rng.integers(0, 6)), replace=False):
                H[i, j] = np.roll(H[i - 1, j], (int(rng.integers(-2, 3)), int(rng.integers(-2, 3))), axis=(0, 1))
    return H, ip, inx, synth.boxes_xyxy(n, seed=21), rng


def next_features(clustered: bool):
    """next.npz `clu_X` / `iid_X`: (400, 256) fp32 embeddings."""
    return _synth().embeddings(400, d=256, seed=31 + clustered, clustered=clustered)


def peaks_inputs():
    """peaks.npz: six generated frames and two built for the MPE / Margin edge cases."""
    synth = _synth()
    rng = np.random.default_rng(33)
    H = synth.heatmaps(6, seed=33)
    e = np.zeros((2, 17, 64, 48), np.float32)
    f = e[0]
    f[0] = 0.25                                                   # constant map: trivial image, no peak
    f[1, 20, 20] = 1; f[1, 20, 24] = 1; f[1, 20, 25] = 0.9          # equal peaks 4 apart: the second is rejected
    f[2, 20, 20] = 1; f[2, 20, 25] = 1                              # equal peaks 5 apart: both kept, margin 0
    f[3, 4, 10] = 2; f[3, 30, 4] = 2; f[3, 59, 10] = 2; f[3, 30, 30] = 0.5   # border peaks are excluded
    f[4, 10:13, 10:13] = 0.7; f[4, 40, 30] = 0.7                    # plateau: every plateau pixel is a candidate
    f[5] = rng.normal(0, 0.02, (64, 48)).astype(np.float32)         # pure noise: more than five candidates
    f[6] = -np.abs(rng.normal(0, 0.02, (64, 48))).astype(np.float32) - 1    # all negative
    f[7, 5, 5] = 1; f[7, 58, 42] = 0.5                              # first / last interior pixel
    f[8, 30, 20] = 1                                                # a single peak: entropy(softmax([x])) = 0
    e[1] = H[0] * 0 + rng.normal(0, 1e-3, (17, 64, 48)).astype(np.float32)
    return np.concatenate([H, e], axis=0)


def coreset_features():
    """coreset.npz: the fp32 feature matrix of every case, by case tag."""
    synth = _synth()
    Xc = synth.embeddings(600, d=256, seed=2, clustered=True)
    Xi = synth.embeddings(500, d=256, seed=4, clustered=False)
    Xd = Xi.copy()
    Xd[100:110] = Xd[10:20]                                       # duplicate rows
    return {"clustered_round0": Xc, "clustered_lab20": Xc, "iid_round0_moks": Xi, "iid_fixed_lambda": Xi,
            "iid_dist_only": Xi, "duplicates": Xd, "zero_unc": Xc,
            "d2048": synth.embeddings(160, d=2048, seed=6, clustered=True)}
