"""CPU oracle of the Macenko stain normalisation -- TEST INFRASTRUCTURE, NOT PRODUCT.

``estimate_literal`` / ``normalize_literal`` restate torchstain's ``NumpyMacenkoNormalizer`` (a port of HEnorm_python) with
``lstsq``, ``eigh``, ``percentile`` and ``exp``, except that the stain matrix is estimated once (from a slide thumbnail)
and then applied to other images.  ``normalizer_matrix`` / ``apply`` are the exact fast form the CUDA kernels compute
(``csrc/stain.cu``): one 3x3 matrix ``M`` formed by a fixed sequence of fp64 operations, and a per-channel threshold
count over the optical-density table instead of ``exp``.  ``tests/test_stain_cpu.py`` checks the fast form against the
literal one over all 2^24 colours; ``tests/test_stain_gpu.py`` compares the kernels with both.
"""
from __future__ import annotations

import numpy as np

IO, ALPHA, BETA = 240, 1.0, 0.15
HE_REF = np.array([[0.5626, 0.2159], [0.7201, 0.8012], [0.4062, 0.5581]])   # torchstain's target
MAXC_REF = np.array([1.9705, 1.0308])


def od_table(io: int = IO) -> np.ndarray:
    """fp64 [256]: ``od[v] = -log((v + 1) / Io)``, strictly decreasing."""
    return -np.log((np.arange(256, dtype=np.float64) + 1) / io)


def _he_of(E: np.ndarray, od_hat: np.ndarray, alpha: float) -> np.ndarray:
    """Steps 4-6: the H-first stain matrix [3, 2] from the two principal eigenvectors ``E`` [3, 2]."""
    T = od_hat.dot(E)
    phi = np.arctan2(T[:, 1], T[:, 0])
    min_phi, max_phi = np.percentile(phi, alpha), np.percentile(phi, 100 - alpha)
    v_min = E.dot(np.array([np.cos(min_phi), np.sin(min_phi)]))
    v_max = E.dot(np.array([np.cos(max_phi), np.sin(max_phi)]))
    return np.array((v_min, v_max)).T if v_min[0] > v_max[0] else np.array((v_max, v_min)).T


def estimate_literal(img: np.ndarray, io: int = IO, alpha: float = ALPHA, beta: float = BETA, flip=(False, False)):
    """torchstain's ``__compute_matrices`` of a uint8 ``[..., 3]`` image: ``(HE [3, 2], maxC [2], n_hat)``, or ``None`` where
    the CUDA estimate reports ``valid = 0`` (fewer than two pixels in ODhat, a singular ``HE^T HE``, a non-finite value or
    ``maxC <= 0``).  ``flip`` negates the eigenvectors, which must not change the result."""
    I = img.reshape(-1, 3)
    OD = -np.log((I.astype(np.float64) + 1) / io)
    od_hat = OD[~np.any(OD < beta, axis=1)]
    n_hat = len(od_hat)
    if n_hat < 2:
        return None
    _, eigvecs = np.linalg.eigh(np.cov(od_hat.T))
    E = eigvecs[:, 1:3].copy()
    for k in range(2):
        if flip[k]:
            E[:, k] = -E[:, k]
    HE = _he_of(E, od_hat, alpha)
    G = HE.T @ HE
    if not G[0, 0] * G[1, 1] - G[0, 1] * G[0, 1] > 0:
        return None
    C = np.linalg.lstsq(HE, OD.T, rcond=None)[0]
    max_c = np.array([np.percentile(C[0, :], 99), np.percentile(C[1, :], 99)])
    if not (np.all(np.isfinite(HE)) and np.all(np.isfinite(max_c)) and np.all(max_c > 0)):
        return None
    return HE, max_c, n_hat


def normalize_literal(img: np.ndarray, he: np.ndarray, max_c: np.ndarray, he_ref=HE_REF, max_c_ref=MAXC_REF, io: int = IO):
    """torchstain's ``normalize`` of a uint8 ``[..., 3]`` image with the given source ``(HE, maxC)`` (no re-estimation)."""
    shape = img.shape
    I = img.reshape(-1, 3)
    OD = -np.log((I.astype(np.float64) + 1) / io)
    C = np.linalg.lstsq(he, OD.T, rcond=None)[0]
    C2 = C / (max_c / max_c_ref)[:, None]
    out = np.multiply(io, np.exp(-he_ref.dot(C2)))
    out[out > 255] = 255
    return out.T.reshape(shape).astype(np.uint8)


def pinv_fixed(he: np.ndarray):
    """``(P, det)``: ``P = (HE^T HE)^-1 HE^T`` [2, 3] by the fixed sequence of the kernels (rows summed 0, 1, 2; every
    product and sum rounded on its own, no FMA)."""
    h = [[float(he[r, c]) for c in range(2)] for r in range(3)]
    g = [[(h[0][i] * h[0][j] + h[1][i] * h[1][j]) + h[2][i] * h[2][j] for j in range(2)] for i in range(2)]
    det = g[0][0] * g[1][1] - g[0][1] * g[0][1]
    inv = [[g[1][1] / det, -g[0][1] / det], [-g[0][1] / det, g[0][0] / det]]
    P = np.array([[inv[i][0] * h[j][0] + inv[i][1] * h[j][1] for j in range(3)] for i in range(2)])
    return P, det


def normalizer_matrix(he: np.ndarray, max_c: np.ndarray, he_ref=HE_REF, max_c_ref=MAXC_REF) -> np.ndarray:
    """fp64 [3, 3]: ``M = HERef diag(maxCRef / maxC) P`` by the fixed sequence of ``k_stain_normalizer``."""
    P, _ = pinv_fixed(he)
    s = [float(max_c_ref[0]) / float(max_c[0]), float(max_c_ref[1]) / float(max_c[1])]
    return np.array([[(float(he_ref[c, 0]) * s[0]) * P[0, j] + (float(he_ref[c, 1]) * s[1]) * P[1, j] for j in range(3)]
                     for c in range(3)])


def apply(img: np.ndarray, M: np.ndarray, od: np.ndarray) -> np.ndarray:
    """The fast form: ``y_c = (M[c,0] od[r] + M[c,1] od[g]) + M[c,2] od[b]`` (products rounded, no FMA), and
    ``out_c = #{v in 0..254 : y_c <= od[v]}``, which equals ``uint8(min(255, Io exp(-y_c)))``."""
    I = img.reshape(-1, 3)
    asc = od[:255][::-1]
    out = np.empty(I.shape, np.uint8)
    for c in range(3):
        A = [M[c, j] * od for j in range(3)]          # the per-CTA tables of the kernel: A[c][j][v] = M[c][j] * od[v]
        y = (A[0][I[:, 0]] + A[1][I[:, 1]]) + A[2][I[:, 2]]
        out[:, c] = 255 - np.searchsorted(asc, y, side="left")
    return out.reshape(img.shape)


def all_colours(lo: int = 0, hi: int = 1 << 24) -> np.ndarray:
    """uint8 [hi - lo, 3]: colours ``lo .. hi-1`` as (r, g, b) = (c >> 16, c >> 8, c) bytes."""
    c = np.arange(lo, hi, dtype=np.uint32)
    return np.stack([(c >> 16) & 255, (c >> 8) & 255, c & 255], axis=1).astype(np.uint8)


def he_image(seed: int, h: int, w: int, he_true: np.ndarray, background: float = 0.3, io: int = IO, noise: float = 1.5,
             shape: float = 2.0, scale: float = 0.35) -> np.ndarray:
    """uint8 [h, w, 3] Beer-Lambert H&E image: ``Io exp(-HE C) + noise``, with gamma-distributed concentrations ``C`` and a
    ``background`` fraction of pixels left without stain (white glass)."""
    rng = np.random.default_rng(seed)
    he = np.asarray(he_true, dtype=np.float64)
    he = he / np.linalg.norm(he, axis=0)
    n = h * w
    C = rng.gamma(shape, scale, size=(2, n)) * (rng.random(n) >= background)
    I = io * np.exp(-(he @ C)) + rng.normal(0, noise, size=(3, n))
    return np.ascontiguousarray(np.clip(I, 0, 255).astype(np.uint8).T.reshape(h, w, 3))


HE_TRUE = np.array([[0.65, 0.07], [0.70, 0.99], [0.29, 0.11]])     # haematoxylin, eosin (normalised in he_image)
HE_TRUE_B = np.array([[0.55, 0.15], [0.78, 0.93], [0.30, 0.33]])   # a second centre's staining
