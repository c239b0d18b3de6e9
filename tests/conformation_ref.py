"""Conformation sampling restated in numpy (DESIGN.md §13, include/polymc.h "conformation sampling").

TEST INFRASTRUCTURE ONLY.  One sample of one chain adds to a row of cols = 8 + 3n + B sums:
  0: 1 · 1–6: S_xx S_yy S_zz S_xy S_xz S_yz of S = (1/n) Σ_i (x_i − x̄)(x_i − x̄)ᵀ · 7: (tr S)²
  8 + s: C_s = Σ_{i=0}^{n−1−s} n̂_i·n̂_{i+s} · 8 + n + i: n̂z_i · 8 + 2n + i: n̂z_i² · 8 + 3n + k: histogram of ζ = r_z/(n b)
with x_i = b (Σ_{k≤i} n̂_k − n̂_i/2) the monomer centres and r = x_{n−1} + (b/2) n̂_{n−1}.  The count, the profile and
the histogram are one IEEE addition per sample (numpy float64 scalars contract nothing), so `Sums.add` reproduces the
device's bits for them; the histogram's bin also needs the device's r_z, which callers may pass (pmc_observables).
`magnitudes` gives, per column, the sum of the magnitudes of the terms, the scale of the rounding of the other sums.
"""
import numpy as np


def centres(nhat, b):
    nhat = np.asarray(nhat, dtype=np.float64)
    return b * (np.cumsum(nhat, axis=0) - 0.5 * nhat)


def bin_of(rz, n, b, bins):
    """bin k = min(B−1, max(0, ⌊(ζ+1)·B/2⌋)), ζ = r_z/(n b), in the device's order of IEEE operations."""
    zeta = np.float64(rz) / (np.float64(n) * np.float64(b))
    u = (zeta + np.float64(1.0)) * np.float64(bins) * np.float64(0.5)
    if u < 1.0:
        return 0
    if u >= bins - 1:
        return bins - 1
    return int(np.floor(u))


def lag_sums(nhat):
    """C_s for s = 0 … n−1 (and Σ|terms| per lag)."""
    nhat = np.asarray(nhat, dtype=np.float64)
    n = nhat.shape[0]
    c, a = np.empty(n), np.empty(n)
    for s in range(n):
        t = nhat[: n - s] * nhat[s:]
        c[s] = t.sum()
        a[s] = np.abs(t).sum()
    return c, a


def sample(nhat, b, bins, rz=None):
    """-> (row of one sample, Σ|terms| per column)."""
    nhat = np.asarray(nhat, dtype=np.float64)
    n = nhat.shape[0]
    x = centres(nhat, b)
    d = x - x.mean(axis=0)
    pairs = [(0, 0), (1, 1), (2, 2), (0, 1), (0, 2), (1, 2)]
    S = np.array([(d[:, i] * d[:, j]).sum() / n for i, j in pairs])
    Sa = np.array([np.abs(d[:, i] * d[:, j]).sum() / n for i, j in pairs])
    row, mag = np.zeros(8 + 3 * n + bins), np.zeros(8 + 3 * n + bins)
    row[0] = 1.0
    row[1:7], mag[1:7] = S, Sa + np.abs(x).sum() * np.abs(x).max() / n   # the centroid's rounding enters every term
    tr = S[:3].sum()
    row[7], mag[7] = tr * tr, 2 * abs(tr) * mag[1:4].sum() + tr * tr
    row[8:8 + n], mag[8:8 + n] = lag_sums(nhat)
    row[8 + n:8 + 2 * n] = nhat[:, 2]
    row[8 + 2 * n:8 + 3 * n] = nhat[:, 2] * nhat[:, 2]
    if bins:
        if rz is None:
            rz = x[n - 1, 2] + 0.5 * b * nhat[n - 1, 2]
        row[8 + 3 * n + bin_of(rz, n, b, bins)] = 1.0
    return row, mag


class Sums:
    """The running sums of one chain, added sample by sample in the device's order."""

    def __init__(self, n, bins):
        self.n, self.bins = n, bins
        self.row = np.zeros(8 + 3 * n + bins)
        self.mag = np.zeros(8 + 3 * n + bins)

    def add(self, nhat, b, rz=None):
        r, m = sample(nhat, b, self.bins, rz)
        n = self.n
        exact = np.zeros(r.shape, bool)
        exact[0] = True
        exact[8 + n:] = True
        # the exact columns: one IEEE addition per sample, element by element
        self.row[exact] = self.row[exact] + r[exact]
        self.row[~exact] += r[~exact]
        self.mag += m


def hand_chains():
    """Hand-built chains with known answers: (name, n̂ [n][3], b, dict of expected averages)."""
    out = []
    n = 7
    rod = np.tile([0.0, 0.0, 1.0], (n, 1))                           # straight rod along z
    out.append(("rod", rod, 1.0, {"Szz": (n * n - 1) / 12.0, "C": np.arange(n, 0, -1).astype(float), "zeta": 1.0}))
    zig = np.array([[np.sin(0.3) * (-1) ** i, 0.0, np.cos(0.3)] for i in range(8)])   # zig-zag in the x–z plane
    c2 = np.cos(0.6)   # n̂_i·n̂_{i+1} = cos²0.3 − sin²0.3
    out.append(("zigzag", zig, 2.0, {"C": np.array([(8 - s) * (1.0 if s % 2 == 0 else c2) for s in range(8)]),
                                      "zeta": np.cos(0.3)}))
    phi = np.linspace(0.0, np.pi, 9)                                  # planar: a half circle, n̂ = (cosϕ, 0, sinϕ)
    pl = np.stack([np.cos(phi), np.zeros_like(phi), np.sin(phi)], axis=1)
    out.append(("planar", pl, 1.0, {"Syy": 0.0, "C": np.array([np.cos(s * np.pi / 8) * (9 - s) for s in range(9)]),
                                    "zeta": np.sin(phi).sum() / 9}))
    return out
