"""Philox4x32-10 and fp64 restatements of the counter-based samplers, shared by the tests.

Every sampling kernel of the library is a short deterministic function of Philox4x32-10 words (key = seed, counter =
(ctr_lo, ctr_hi) as two 64-bit halves), so each draw can be recomputed on the host:

- `ref_base_sample` restates `base_sample_kernel` (csrc/elementwise.cuh): Laplace by inverse CDF, Normal by Box-Muller.
- `ref_radial_sample` restates `radial_sample_kernel` (csrc/radial.cuh): mixture component, Marsaglia-Tsang rejection
  rounds, the `a < 1` boost, the generalised-Gamma power, log-normal radii, and the direction on the unit Lp sphere.

Both evaluate everything after the integer words in fp64.  The radial sampler takes discrete decisions on fp32 values
(which mixture component, whether a rejection round accepts); `ref_radial_sample` flags a row as *fragile* when one of
those decisions lies so close to its threshold that fp32 and fp64 may decide differently.
"""
from types import SimpleNamespace

import numpy as np

from usflows_b200 import ops

MASK = np.uint64(0xFFFFFFFF)
U64 = (1 << 64) - 1
RTAG = 1 << 62                 # radius sub-stream tag of radial_sample_kernel
NTAG = 1 << 63                 # second Box-Muller stream of base_sample_kernel
EXTREMAL_STREAM = 0x100        # p = inf: sub-stream of the pinned coordinate
F32_THIRD = float(np.float32(1.0) / np.float32(3.0))


def np_philox4x32_10(ctr, key):
    """Philox4x32-10 on uint64 arrays holding 32-bit words: ctr = 4 arrays, key = 2 arrays (or scalars)."""
    c0, c1, c2, c3 = (np.asarray(c, dtype=np.uint64) & MASK for c in ctr)
    k0, k1 = (np.asarray(k, dtype=np.uint64) & MASK for k in key)
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c0
        p1 = np.uint64(0xCD9E8D57) * c2
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & MASK, (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & MASK
        k0 = (k0 + np.uint64(0x9E3779B9)) & MASK
        k1 = (k1 + np.uint64(0xBB67AE85)) & MASK
    return c0, c1, c2, c3


def philox(seed: int, ctr_lo, ctr_hi: int):
    """The four words of Philox4x32-10(seed, (ctr_lo, ctr_hi)) as the kernels call it: ctr_lo an array of 64-bit
    counters, ctr_hi one 64-bit value (taken modulo 2^64, as the kernels' uint64_t arithmetic does)."""
    lo = np.asarray(ctr_lo, dtype=np.uint64)
    hi = int(ctr_hi) & U64
    seed = int(seed) & U64
    return np_philox4x32_10((lo & MASK, lo >> np.uint64(32), np.uint64(hi & 0xFFFFFFFF), np.uint64(hi >> 32)),
                            (np.uint64(seed & 0xFFFFFFFF), np.uint64(seed >> 32)))


def u01(w):
    """u01_open: 23 random bits + 1/2, scaled into (0, 1); exact in fp32 and fp64."""
    return ((w >> np.uint64(9)).astype(np.float64) + 0.5) * 2.0 ** -23


def _box_muller(w_rad, w_ang):
    rad = np.sqrt(-2.0 * np.log(u01(w_rad)))
    ang = 2.0 * np.pi * u01(w_ang)
    return rad * np.cos(ang), rad * np.sin(ang)


# ---- Laplace / Normal base ---------------------------------------------------------------------------------------------
def ref_base_eps(rows: int, d: int, kind: int, seed: int, offset: int) -> np.ndarray:
    """Standardised draws e [rows, d] of base_sample_kernel: group g of row r uses counter (r * ceil(d / 4) + g, offset)."""
    d4 = (d + 3) // 4
    i = np.arange(rows * d4, dtype=np.uint64)
    w = philox(seed, i, offset)
    if kind == ops.BASE_LAPLACE:
        e = []
        for t in range(4):
            u = 2.0 * u01(w[t]) - 1.0
            e.append(-np.sign(u) * np.log1p(-np.abs(u)))
    else:
        w2 = philox(seed, i, int(offset) ^ NTAG)
        e0, e1 = _box_muller(w[0], w2[0])
        e2, e3 = _box_muller(w[2], w2[2])
        e = [e0, e1, e2, e3]
    return np.stack(e, axis=-1).reshape(rows, d4 * 4)[:, :d]


def ref_base_sample(rows: int, d: int, loc, scale, kind: int, seed: int, offset: int) -> np.ndarray:
    """fp64 values [rows, d] of usf_base_sample: loc[j] + scale[j] * e[r, j]."""
    loc = np.asarray(loc, dtype=np.float64).reshape(-1)
    scale = np.asarray(scale, dtype=np.float64).reshape(-1)
    return loc[None, :] + scale[None, :] * ref_base_eps(rows, d, kind, seed, offset)


# ---- Lp-radial base ----------------------------------------------------------------------------------------------------
def unpack_norm_params(kind: int, K: int, params):
    """The packed radius parameters (layout of USF_NORM_*) as fp64 arrays: dict of logits / a / b / scale / power."""
    p = np.asarray(params, dtype=np.float32).astype(np.float64).reshape(-1)
    if kind == ops.NORM_LOGNORMAL:
        return dict(mu=p[0:1], sigma=p[1:2])
    out = dict(logits=p[:K], a=p[K:2 * K], b=p[2 * K:3 * K])
    if kind == ops.NORM_GENGAMMA_MIXTURE:
        out.update(scale=p[3 * K:4 * K], power=p[4 * K:5 * K])
    return out


def mixture_cdf(logits) -> np.ndarray:
    w = np.exp(logits - logits.max())
    return np.cumsum(w / w.sum())


def _gamma_mt(a32, seed, rows_idx, off, fragile):
    """Marsaglia-Tsang Gamma(a, 1) draws for the rows `rows_idx` (a32 [n]: fp32 shapes >= 1), rounds at counters
    (r, off + 2 + it).  Marks in `fragile` (indexed like rows_idx) rows whose decisions sit on a threshold."""
    n = rows_idx.shape[0]
    dd = (a32.astype(np.float32) - np.float32(F32_THIRD)).astype(np.float64)   # the kernel forms a - 1/3 in fp32
    c = 1.0 / np.sqrt(9.0 * dd)
    out = dd.copy()
    todo = np.ones(n, dtype=bool)
    for it in range(64):
        if not todo.any():
            break
        idx = np.nonzero(todo)[0]
        w = philox(seed, rows_idx[idx].astype(np.uint64), (off + 2 + it) & U64)
        x = np.sqrt(-2.0 * np.log(u01(w[0]))) * np.cos(2.0 * np.pi * u01(w[1]))
        v0 = 1.0 + c[idx] * x
        # v0 <= 0: the kernel's v0 carries one rounding of c * x (|c x| < 1 there)
        fragile[idx] |= np.abs(v0) < 1e-6
        ok = v0 > 0
        v = np.where(ok, v0, 1.0) ** 3
        lhs = np.log(u01(w[2]))
        d_ = dd[idx]
        rhs = 0.5 * x * x + d_ - d_ * v + d_ * np.log(v)
        # the fp32 right-hand side cancels terms of size dd: its rounding error scales with them
        margin = 2.0 ** -22 * (0.5 * x * x + d_ + d_ * v + d_ * np.abs(np.log(v))) + 1e-6
        fragile[idx] |= ok & (np.abs(lhs - rhs) < margin)
        acc = ok & (lhs < rhs)
        out[idx[acc]] = (d_ * v)[acc]
        todo[idx[acc]] = False
    return out


def ref_radial_sample(rows: int, d: int, loc, p_kind: int, kind: int, params, K: int, seed: int, offset: int,
                      chunk: int = 4096):
    """fp64 restatement of usf_radial_sample.  Returns a namespace with
    x [rows, d] (the samples), radius [rows], nrm [rows] (the Lp norm of the raw direction draws; 1 for p = inf),
    extremal [rows] (p = inf: the pinned coordinate, else -1) and fragile [rows] (bool: a discrete decision of the row lies
    within rounding distance of its threshold -- the mixture component, v0 <= 0, or a rejection round's accept test)."""
    seed, offset = int(seed) & U64, int(offset) & U64
    loc = np.asarray(loc, dtype=np.float64).reshape(-1)
    if loc.size == 1 and d > 1:
        loc = np.full(d, loc[0])
    P = unpack_norm_params(kind, K, params)
    r_idx = np.arange(rows, dtype=np.uint64)
    off_r = offset ^ RTAG
    fragile = np.zeros(rows, dtype=bool)
    if kind == ops.NORM_LOGNORMAL:
        w = philox(seed, r_idx, off_r)
        z, _ = _box_muller(w[0], w[1])
        radius = np.exp(P["mu"][0] + P["sigma"][0] * z)
    else:
        w = philox(seed, r_idx, off_r)
        u = u01(w[0])
        cdf = mixture_cdf(P["logits"])
        k = np.minimum(np.searchsorted(cdf[:-1], u, side="left"), K - 1) if K > 1 else np.zeros(rows, dtype=np.int64)
        if K > 1:       # fp32 cumulative weights: a few roundings of each partial sum
            th = cdf[:-1]
            margin = 2.0 ** -21 * th + 2.0 ** -23 * np.sqrt(np.arange(1, K))
            fragile |= (np.abs(u[:, None] - th[None, :]) < margin[None, :]).any(axis=1)
        a, b = P["a"][k], P["b"][k]
        if kind == ops.NORM_LOGNORMAL_MIXTURE:                      # a = mu_k, b = sigma_k
            w1 = philox(seed, r_idx, (off_r + 1) & U64)
            z, _ = _box_muller(w1[0], w1[1])
            radius = np.exp(a + b * z)
        else:
            boost = a < 1.0
            a32 = a.astype(np.float32)
            shape = np.where(boost, (a32 + np.float32(1.0)).astype(np.float64), a)      # a + 1.f in fp32
            fr = np.zeros(rows, dtype=bool)
            g = _gamma_mt(shape, seed, r_idx, (off_r + 1) & U64, fr)
            fragile |= fr
            inv_a = (np.float32(1.0) / a32).astype(np.float64)                           # 1.f / a in fp32
            g = np.where(boost, g * np.power(u01(w[1]), np.where(boost, inv_a, 1.0)), g)
            radius = g / b
            if kind == ops.NORM_GENGAMMA_MIXTURE:                                         # R = s_k S^(1 / q_k)
                q = P["power"][k]
                inv_q = (np.float32(1.0) / q.astype(np.float32)).astype(np.float64)
                radius = P["scale"][k] * np.where(q == 2.0, np.sqrt(radius), np.power(radius, inv_q))
    extremal = np.full(rows, -1, dtype=np.int64)
    if p_kind == ops.LP_INF:
        w = philox(seed, r_idx, (off_r + EXTREMAL_STREAM) & U64)
        # u * d is exact in fp64; the kernel rounds it once to fp32 before the truncation
        extremal = np.minimum(d - 1, np.floor(np.float32(u01(w[0]) * d).astype(np.float64)).astype(np.int64))
    d4 = (d + 3) // 4
    x = np.empty((rows, d))
    nrm = np.ones(rows)
    for r0 in range(0, rows, chunk):
        r1 = min(rows, r0 + chunk)
        ctr = (np.arange(r0, r1, dtype=np.uint64)[:, None] * np.uint64(d4) + np.arange(d4, dtype=np.uint64)[None, :])
        w = philox(seed, ctr, offset)
        if p_kind == ops.LP_2:
            e0, e1 = _box_muller(w[0], w[1])
            e2, e3 = _box_muller(w[2], w[3])
            e = np.stack([e0, e1, e2, e3], axis=-1)
        elif p_kind == ops.LP_1:
            e = np.stack([np.where(w[t] & np.uint64(1), 1.0, -1.0) * np.log(u01(w[t])) for t in range(4)], axis=-1)
        else:
            e = np.stack([2.0 * u01(w[t]) - 1.0 for t in range(4)], axis=-1)
        e = e.reshape(r1 - r0, d4 * 4)[:, :d]
        if p_kind == ops.LP_2:
            nrm[r0:r1] = np.sqrt((e * e).sum(axis=1))
        elif p_kind == ops.LP_1:
            nrm[r0:r1] = np.abs(e).sum(axis=1)
        else:
            e[np.arange(r1 - r0), extremal[r0:r1]] = 1.0
        x[r0:r1] = loc[None, :] + (radius[r0:r1] / nrm[r0:r1])[:, None] * e
    return SimpleNamespace(x=x, radius=radius, nrm=nrm, extremal=extremal, fragile=fragile)
