"""NumPy restatement of the scrambled Sobol' variates of the tolerance-study sampling contract
(include/okin.h, DESIGN.md section 10), written from the definition alone: the Joe-Kuo direction
numbers expanded to 52 bits from SciPy's npz, the Gray-code point order, the linear matrix scramble
and digital shift drawn with Philox, and Wichura's AS241 inverse normal CDF."""

from __future__ import annotations

import os

import numpy as np

import study_reference as ref

BITS = 52
SOBOL_UNIFORM, SOBOL_NORMAL = 3, 4
MASK52 = (1 << BITS) - 1


def scipy_table() -> tuple:
    import scipy.stats
    with np.load(os.path.join(os.path.dirname(scipy.stats.__file__), "_sobol_direction_numbers.npz")) as f:
        return np.asarray(f["poly"], np.int64), np.asarray(f["vinit"], np.int64)


def directions(n_dims: int) -> np.ndarray:
    """``V [n_dims, 52]`` uint64: direction number ``k`` of each dimension, bit 51 = the 2^-1 digit."""
    poly, vinit = scipy_table()
    V = np.zeros((n_dims, BITS), np.uint64)
    for d in range(n_dims):
        p = int(poly[d])
        m = p.bit_length() - 1
        mk = []
        for k in range(BITS):
            if d == 0:
                x = 1
            elif k < m:
                x = int(vinit[d, k])
            else:
                x = mk[k - m]
                for l in range(1, m + 1):
                    if (p >> (m - l)) & 1:
                        x ^= mk[k - l] << l
            mk.append(x)
        V[d] = [x << (BITS - 1 - k) for k, x in enumerate(mk)]
    return V


def scramble_word(seed: int, v: int, a) -> np.ndarray:
    """``W(a)``: bits 63..12 of the first 64-bit word of Philox at counter (a, 0, v, 1)."""
    a = np.atleast_1d(np.asarray(a, np.uint64))
    x = ref.philox4x32_10([a, np.zeros_like(a), np.full_like(a, v), np.ones_like(a)],
                          (seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF))
    return ((x[1] << np.uint64(32)) | x[0]) >> np.uint64(64 - BITS)


def scramble(seed: int, v: int) -> tuple:
    """``(rows [52], shift)`` of Sobol' variate ``v``: row k of the lower-triangular matrix M_v."""
    w = scramble_word(seed, v, np.arange(BITS + 1))
    rows = []
    for k in range(BITS):
        diag = 1 << (BITS - 1 - k)
        rows.append((int(w[k]) & ~(diag - 1)) | diag)
    return np.array(rows, np.uint64), int(w[BITS])


def apply_matrix(rows: np.ndarray, x: np.ndarray) -> np.ndarray:
    """``M x`` for a uint64 array ``x``: digit k (bit 51 - k) is the parity of ``rows[k] & x``."""
    y = np.zeros_like(x)
    for k in range(BITS):
        bit = np.bitwise_count(x & rows[k]).astype(np.uint64) & np.uint64(1)
        y |= bit << np.uint64(BITS - 1 - k)
    return y


def points(V: np.ndarray, j) -> np.ndarray:
    """Unscrambled integers ``X [n, len(V)]`` of the points ``j``: XOR of V[d][k] over the set bits of gray(j)."""
    j = np.asarray(j, np.uint64)
    g = j ^ (j >> np.uint64(1))
    X = np.zeros((j.size, V.shape[0]), np.uint64)
    for k in range(BITS):
        on = ((g >> np.uint64(k)) & np.uint64(1)).astype(bool)
        X[on] ^= V[:, k][None, :]
    return X


def scrambled_points(seed: int, variate_ids, V: np.ndarray, j) -> np.ndarray:
    """``X [n, len(variate_ids)]``: Sobol' variate ``variate_ids[d]`` takes dimension ``d``."""
    X = points(V[:len(variate_ids)], j)
    for d, v in enumerate(variate_ids):
        rows, shift = scramble(seed, v)
        X[:, d] = apply_matrix(rows, X[:, d]) ^ np.uint64(shift)
    return X


# AS241 (PPND16) coefficients, highest degree last
A = [3.3871328727963666080e0, 1.3314166789178437745e+2, 1.9715909503065514427e+3, 1.3731693765509461125e+4,
     4.5921953931549871457e+4, 6.7265770927008700853e+4, 3.3430575583588128105e+4, 2.5090809287301226727e+3]
B = [1.0, 4.2313330701600911252e+1, 6.8718700749205790830e+2, 5.3941960214247511077e+3,
     2.1213794301586595867e+4, 3.9307895800092710610e+4, 2.8729085735721942674e+4, 5.2264952788528545610e+3]
C = [1.42343711074968357734e0, 4.63033784615654529590e0, 5.76949722146069140550e0, 3.64784832476320460504e0,
     1.27045825245236838258e0, 2.41780725177450611770e-1, 2.27238449892691845833e-2, 7.74545014278341407640e-4]
D = [1.0, 2.05319162663775882187e0, 1.67638483018380384940e0, 6.89767334985100004550e-1,
     1.48103976427480074590e-1, 1.51986665636164571966e-2, 5.47593808499534494600e-4, 1.05075007164441684324e-9]
E = [6.65790464350110377720e0, 5.46378491116411436990e0, 1.78482653991729133580e0, 2.96560571828504891230e-1,
     2.65321895265761230930e-2, 1.24266094738807843860e-3, 2.71155556874348757815e-5, 2.01033439929228813265e-7]
F = [1.0, 5.99832206555887937690e-1, 1.36929880922735805310e-1, 1.48753612908506148525e-2,
     7.86869131145613259100e-4, 1.84631831751005468180e-5, 1.42151175831644588870e-7, 2.04426310338993978564e-15]


def _horner(c, r):
    y = np.full_like(r, c[-1])
    for a in c[-2::-1]:
        y = y * r + a
    return y


def ppnd16(p) -> np.ndarray:
    """Wichura's AS241: the standard normal quantile of ``p`` in (0, 1)."""
    p = np.asarray(p, np.float64)
    q = p - 0.5
    central = np.abs(q) <= 0.425
    r0 = 0.180625 - q * q
    z_c = q * _horner(A, r0) / _horner(B, r0)
    with np.errstate(divide="ignore", invalid="ignore"):
        r = np.sqrt(-np.log(np.where(q < 0, p, 1.0 - p)))
    near = r - 1.6
    far = r - 5.0
    z_t = np.where(r <= 5.0, _horner(C, near) / _horner(D, near), _horner(E, far) / _horner(F, far))
    return np.where(central, z_c, np.where(q < 0, -z_t, z_t))


def variates(kind, levels, seed: int, ids) -> np.ndarray:
    """``z [n_ids, n_variates]`` of the instances ``ids`` under the full contract (Philox, grid, Sobol')."""
    kind = [int(k) for k in kind]
    ids = np.asarray(ids, np.uint64)
    z = ref.variates([k if k < 3 else 0 for k in kind], levels, seed, ids)
    sob = [v for v, k in enumerate(kind) if k in (SOBOL_UNIFORM, SOBOL_NORMAL)]
    if not sob:
        return z
    period = 1
    for v, k in enumerate(kind):
        if k == 2:
            period *= int(levels[v])
    assert period < 2 ** 63
    X = scrambled_points(seed, sob, directions(len(sob)), ids // np.uint64(period))
    for d, v in enumerate(sob):
        if kind[v] == SOBOL_UNIFORM:
            z[:, v] = X[:, d].astype(np.float64) * 2.0 ** -51 - 1.0
        else:
            z[:, v] = ppnd16((2 * X[:, d] + np.uint64(1)).astype(np.float64) * 2.0 ** -53)
    return z


def inputs(tables: dict, seed: int, ids) -> np.ndarray:
    """``[n_ids, n_coords]``: nominal + scale * z[source], nominal where source = -1."""
    z = variates(tables["variate_kind"], tables["grid_levels"], seed, ids)
    src = np.asarray(tables["source"])
    out = np.repeat(np.asarray(tables["nominal"], dtype=np.float64)[None, :], len(z), axis=0)
    live = src >= 0
    out[:, live] = tables["scale"][live][None, :] * z[:, src[live]] + tables["nominal"][live][None, :]
    return out
