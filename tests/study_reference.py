"""NumPy restatement of the tolerance-study sampling contract and statistics (include/okin.h,
DESIGN.md section 10), written from the definition alone: Philox4x32-10 on uint64 arrays, the
normal / uniform / grid variates, the coordinate rule, and plain numpy statistics of per-instance
outputs to check a study's reductions against."""

from __future__ import annotations

import numpy as np

M0, M1, W0, W1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57), 0x9E3779B9, 0xBB67AE85
MASK = np.uint64(0xFFFFFFFF)


def philox4x32_10(ctr, key) -> list:
    """Philox4x32-10 of counters ``ctr`` (4 uint arrays) under ``key`` (2 ints): 4 uint64 arrays < 2^32."""
    c = [np.asarray(x, dtype=np.uint64) & MASK for x in ctr]
    k0, k1 = int(key[0]), int(key[1])
    for r in range(10):
        if r:
            k0, k1 = (k0 + W0) & 0xFFFFFFFF, (k1 + W1) & 0xFFFFFFFF
        p0, p1 = M0 * c[0], M1 * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ np.uint64(k0), p1 & MASK, (p0 >> np.uint64(32)) ^ c[3] ^ np.uint64(k1),
             p0 & MASK]
    return c


def cospi(x: np.ndarray) -> np.ndarray:
    """cos(pi x) on [0, 2): exact reduction to [0, 1/4], then cos or sin of pi r."""
    r = np.where(x >= 1.0, 2.0 - x, x)
    sign = np.where(r > 0.5, -1.0, 1.0)
    r = np.where(r > 0.5, 1.0 - r, r)
    return sign * np.where(r > 0.25, np.sin(np.pi * (0.5 - r)), np.cos(np.pi * r))


def variates(kind, levels, seed: int, ids) -> np.ndarray:
    """``z [n_ids, n_variates]`` of the instances ``ids``."""
    ids = np.asarray(ids, dtype=np.uint64)
    key = (seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)
    z = np.zeros((ids.size, len(kind)))
    period = 1
    for v, k in enumerate(kind):
        if k == 2:
            period *= int(levels[v])
    node = ids % np.uint64(period) if period < 2 ** 63 else ids
    place = 1
    for v, k in enumerate(kind):
        if k == 2:
            L = int(levels[v])
            d = (node // np.uint64(place)) % np.uint64(L)
            z[:, v] = d.astype(np.float64) / float(L - 1) * 2.0 - 1.0
            place *= L
            continue
        x = philox4x32_10([ids & MASK, ids >> np.uint64(32), np.full(ids.size, v, np.uint64),
                           np.zeros(ids.size, np.uint64)], key)
        u = (((x[1] << np.uint64(32)) | x[0]) >> np.uint64(11)).astype(np.float64) * 2.0 ** -53
        if k == 1:
            z[:, v] = 2.0 * u - 1.0
        else:
            u2 = (((x[3] << np.uint64(32)) | x[2]) >> np.uint64(11)).astype(np.float64) * 2.0 ** -53
            z[:, v] = np.sqrt(-2.0 * np.log(1.0 - u)) * cospi(2.0 * u2)
    return z


def inputs(tables: dict, seed: int, ids) -> np.ndarray:
    """``[n_ids, n_coords]``: nominal + scale * z[source], nominal where source = -1."""
    z = variates(tables["variate_kind"], tables["grid_levels"], seed, ids)
    src = np.asarray(tables["source"])
    out = np.repeat(np.asarray(tables["nominal"], dtype=np.float64)[None, :], len(z), axis=0)
    live = src >= 0
    out[:, live] = tables["scale"][live][None, :] * z[:, src[live]] + tables["nominal"][live][None, :]
    return out


def statistics(values: np.ndarray, status: np.ndarray, failed_step: np.ndarray, hist_lo=None, hist_hi=None,
               bins: int = 0, id_offset: int = 0) -> dict:
    """Plain numpy statistics of ``values [n, S, Q]`` over the accepted steps (status 0 or step <
    failed_step), finite values counted, non-finite ones in ``nonfinite``."""
    n, S, Q = values.shape
    accepted = (status[:, None] == 0) | (np.arange(S)[None, :] < failed_step[:, None])
    acc = np.broadcast_to(accepted[:, :, None], values.shape)
    fin = np.isfinite(values)
    good = acc & fin
    out = {"count": good.sum(0), "nonfinite": (acc & ~fin).sum(0)}
    mean, std = np.full((S, Q), np.nan), np.full((S, Q), np.nan)
    mn, mx = np.full((S, Q), np.nan), np.full((S, Q), np.nan)
    amin, amax = np.full((S, Q), -1, np.int64), np.full((S, Q), -1, np.int64)
    hist = np.zeros((S, Q, bins + 2), np.int64) if bins else None
    for s in range(S):
        for q in range(Q):
            col = values[good[:, s, q], s, q]
            idx = np.nonzero(good[:, s, q])[0] + id_offset
            if col.size == 0:
                continue
            mean[s, q] = col.mean()
            if col.size >= 2:
                std[s, q] = col.std(ddof=1)
            mn[s, q], mx[s, q] = col[np.argmin(col)], col[np.argmax(col)]
            amin[s, q], amax[s, q] = idx[np.argmin(col)], idx[np.argmax(col)]
            if bins:
                lo, hi = hist_lo[q], hist_hi[q]
                b = np.where(col < lo, 0, np.where(col >= hi, bins + 1, 1 + np.minimum(
                    np.floor((col - lo) / (hi - lo) * bins), bins - 1).astype(np.int64)))
                hist[s, q] = np.bincount(b.astype(np.int64), minlength=bins + 2)
    out.update(mean=mean, std=std, min=mn, max=mx, argmin=amin, argmax=amax, histogram=hist,
               status_counts=np.bincount(status, minlength=4)[:4],
               failed_at_step=np.bincount(failed_step[(failed_step >= 0) & (failed_step < S)], minlength=S)[:S])
    return out


def quantity_values(solver, names, res) -> np.ndarray:
    """``[n, S, Q]`` per-instance values of the study quantities ``names`` from a solve result
    (a ``BatchSweepResult`` or an emulation output dict)."""
    get = (lambda k: res[k]) if isinstance(res, dict) else (lambda k: getattr(res, {"iters": "nfev"}.get(k, k)))
    prog = solver.program
    cols = []
    for name in names:
        if name == "solver_max_residual":
            cols.append(get("max_residual"))
        elif name == "solver_nfev":
            cols.append(get("iters").astype(np.float64))
        elif name in prog.metric_names:
            cols.append(get("metrics")[:, :, prog.metric_names.index(name)])
        else:
            point, axis = name[:-2], "xyz".index(name[-1])
            slot = [k.name.lower() for k in prog.out_keys].index(point)
            cols.append(get("positions")[:, :, slot, axis])
    return np.stack(cols, axis=-1)
