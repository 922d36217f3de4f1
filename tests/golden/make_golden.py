"""Generates tests/golden/*.npz (run once, here, where scipy is installed; outputs are committed).

Why scipy: the reference's own implementation of this path is absent from /root/reference
(raft::distance and pylibraft.distance were removed upstream in 26.02, CHANGELOG.md:59), so the
reference itself cannot be imported to generate vectors.  The historical pylibraft tests compared
against scipy.spatial.distance.cdist (SURVEY.md section 4, [RECALLED]) and BASELINE.json configs[0]
names the same check, so cdist output on seeded inputs is what is pinned here, together with the
known-answer vectors that DO survive in the reference's tests:
  cpp/tests/matrix/argmin.cu:71-75            row-argmin {0,3,3}
  cpp/tests/core/operators_host.cpp:134-152   argmin_op tie-break cases
"""
import os
import numpy as np
from scipy.spatial.distance import cdist

HERE = os.path.dirname(os.path.abspath(__file__))
SCIPY = {"L2Expanded": "sqeuclidean", "L2SqrtExpanded": "euclidean", "CosineExpanded": "cosine",
         "L1": "cityblock", "Linf": "chebyshev", "Canberra": "canberra", "CorrelationExpanded": "correlation"}
# L2Unexpanded / L2SqrtUnexpanded have the same exact values as the expanded forms: stored once, aliased by the
# `golden` fixture in tests/conftest.py (keeps the file under 1 MB)


def blobs(rows, cols, seed, centers=None):
    rng = np.random.default_rng(seed)
    if centers is None:
        centers = rng.uniform(-10, 10, size=(5, cols))
    lab = rng.integers(0, 5, size=rows)
    return (centers[lab] + rng.standard_normal((rows, cols))).astype(np.float32), centers


def main():
    out = {}
    for name, (m, n, k) in {"small": (37, 29, 19), "cfg1": (128, 96, 32)}.items():
        x, c = blobs(m, k, 1234)
        y, _ = blobs(n, k, 4321, c)
        out[f"{name}_x"], out[f"{name}_y"] = x, y
        x64, y64 = x.astype(np.float64), y.astype(np.float64)
        for metric, sp in SCIPY.items():
            out[f"{name}_{metric}"] = cdist(x64, y64, sp)
        out[f"{name}_LpUnexpanded_p3"] = cdist(x64, y64, "minkowski", p=3.0)
        out[f"{name}_InnerProduct"] = x64 @ y64.T
        d = cdist(x64, y64, "sqeuclidean")
        out[f"{name}_nn_idx"] = np.argmin(d, axis=1).astype(np.int32)
        out[f"{name}_nn_val"] = d.min(axis=1)
    # probability-like inputs for the distribution metrics (rows sum to 1, a few exact zeros)
    rng = np.random.default_rng(99)
    px = rng.random((33, 21)); py = rng.random((27, 21))
    px[rng.random(px.shape) < 0.1] = 0.0
    py[rng.random(py.shape) < 0.1] = 0.0
    px = (px / px.sum(1, keepdims=True)).astype(np.float32)
    py = (py / py.sum(1, keepdims=True)).astype(np.float32)
    out["prob_x"], out["prob_y"] = px, py
    p64, q64 = px.astype(np.float64), py.astype(np.float64)
    from scipy.special import rel_entr
    out["prob_KLDivergence"] = 0.5 * np.array([[rel_entr(a, b).sum() for b in q64] for a in p64])  # reference halves the sum
    m_ = 0.5 * (p64[:, None, :] + q64[None, :, :])
    js = 0.5 * (rel_entr(p64[:, None, :], m_).sum(-1) + rel_entr(q64[None, :, :], m_).sum(-1))
    out["prob_JensenShannon"] = np.sqrt(js)           # == scipy jensenshannon for normalised rows
    out["prob_HellingerExpanded"] = np.sqrt(np.maximum(1.0 - np.sqrt(p64) @ np.sqrt(q64).T, 0.0))
    bx = (rng.random((33, 40)) > 0.5).astype(np.float32); by = (rng.random((27, 40)) > 0.5).astype(np.float32)
    out["bool_x"], out["bool_y"] = bx, by
    out["bool_HammingUnexpanded"] = cdist(bx, by, "hamming")
    out["bool_RusselRaoExpanded"] = cdist(bx.astype(bool), by.astype(bool), "russellrao")
    out["bool_JaccardExpanded"] = cdist(bx.astype(bool), by.astype(bool), "jaccard")
    out["bool_DiceExpanded"] = cdist(bx.astype(bool), by.astype(bool), "dice")
    cx = rng.random((33, 40)); cy = rng.random((27, 40))            # non-negative "abundance" vectors
    out["count_x"], out["count_y"] = cx.astype(np.float32), cy.astype(np.float32)
    out["count_BrayCurtis"] = cdist(out["count_x"].astype(np.float64), out["count_y"].astype(np.float64), "braycurtis")
    # reference known answers
    out["ref_argmin_in"] = np.array([0.1, 0.2, 0.3, 0.4, 0.4, 0.3, 0.2, 0.1, 0.2, 0.3, 0.5, 0.0],
                                    dtype=np.float32).reshape(3, 4)   # argmin.cu:71-72
    out["ref_argmin_out"] = np.array([0, 3, 3], dtype=np.int32)
    np.savez_compressed(os.path.join(HERE, "distance_golden.npz"), **out)
    print("wrote", os.path.join(HERE, "distance_golden.npz"), len(out), "arrays")


if __name__ == "__main__":
    main()
