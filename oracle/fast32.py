"""TEST INFRASTRUCTURE ONLY -- a bit-exact numpy restatement of the fp32 fast mode (lsqrrecipes_b200/csrc/fast_forms.cuh).

Every step of that path is deterministic IEEE arithmetic: the per-hypothesis constants are hoisted in fp64 without
contraction (hoist32<M>), the residuals are explicit fma.rn / add.rn / sub.rn / mul.rn on fp32 pairs (Eval<M>), and the
decisions are integer compares on bit patterns (count_carry), |s| < thr (count_abs_lt) or the sign bit (count_sign).  The
functions below restate each step in the kernels' operation order, so the fp32 count of every hypothesis is predicted
exactly, not within a tolerance.

  fma32(a, b, c)               correctly rounded fp32 fused multiply-add
  center_single(model, data)   the centre c of the single-problem path (center_sample_kernel's summation order)
  copy32(model, data, c)       the fp32 copy of the data (ingest_kernel / the batch kernels)
  hoist(model, prm, c, cfg)    hoist32<M> of one parameter vector (NaN row -> hoist32_kernel's degenerate row)
  decisions(...)               per-datum fp32 decision of one hypothesis; counts(...) for many
  replay(...)                  the round loop and stop rule of the batched kernels over given per-hypothesis counts

Also the fp32 rounding band of the threshold (fp32_band) and the float64 residuals it is measured on (residual64).
"""
import math

import numpy as np

from oracle.pyoracle import INFO, MODELS

F32 = np.float32
CNAN = np.uint32(0x7FFFFFFF).view(F32)   # the NaN the GPU produces for every NaN result
_MIDMASK = np.uint64((1 << 29) - 1)      # fp64 mantissa bits below an fp32 normal's last bit
_HALF = np.uint64(1 << 28)
_OVF = 2.0 ** 128 - 2.0 ** 103           # fp32 overflow threshold (ties to even round to inf)
_FLT_MAX = float(np.finfo(np.float32).max)


def _canon(r):
    r = np.asarray(r, dtype=F32)
    return np.where(np.isnan(r), CNAN, r).astype(F32)


def _f32(x):
    """(float) of a double: round to nearest even, NaN canonical."""
    with np.errstate(over="ignore", invalid="ignore"):
        return _canon(np.asarray(x, dtype=np.float64).astype(F32))


# ---- fp32 arithmetic as fma.rn / add.rn / sub.rn / mul.rn -------------------------------------------
def fma32(a, b, c):
    """Correctly rounded a * b + c in fp32.  The product of two fp32 values is exact in fp64; the fp64 sum s is rounded once
    more to fp32, which is right unless s lies exactly on an fp32 rounding boundary (a midpoint, or the overflow threshold)
    and the sum was inexact: there the TwoSum error decides the side.  Subnormal fp32 results take the same test on the
    subnormal grid.  NaN results are canonical."""
    a, b, c = (np.asarray(v, dtype=F32) for v in (a, b, c))
    a, b, c = np.broadcast_arrays(a, b, c)
    a64, b64, c64 = a.astype(np.float64), b.astype(np.float64), c.astype(np.float64)
    with np.errstate(over="ignore", invalid="ignore"):
        p = a64 * b64
        s = p + c64
        r = s.astype(F32)
        finite = np.isfinite(a64) & np.isfinite(b64) & np.isfinite(c64)
        sb = np.abs(s).view(np.uint64)
        # candidates: fp32-normal midpoints (bit 28 set, bits 0..27 clear), anything below the normal range, the overflow edge
        cand = finite & (((sb & _MIDMASK) == _HALF) | (np.abs(s) < 2.0 ** -126) | (np.abs(s) == _OVF))
        if cand.any():
            i = np.flatnonzero(cand.ravel())
            pi, ci, si = p.ravel()[i], c64.ravel()[i], s.ravel()[i]
            bb = si - pi
            e = (pi - (si - bb)) + (ci - bb)          # TwoSum: p + c = s + e exactly
            ri = si.astype(F32)
            r64 = ri.astype(np.float64)
            toward = np.where(si > r64, F32(np.inf), F32(-np.inf))
            other = np.nextafter(ri, toward)
            mid = np.where(np.isinf(ri), np.sign(si) * _OVF, (r64 + other.astype(np.float64)) / 2.0)
            on_mid = (r64 != si) & (si == mid) & (e != 0)
            # the exact value lies beyond the midpoint on e's side: take the neighbour on that side
            go_other = on_mid & (np.sign(e) == np.sign(si - r64))
            ri = np.where(go_other, other, ri)
            # on the midpoint with e pointing back towards r: r is right
            flat = r.ravel().copy()
            flat[i] = ri
            r = flat.reshape(r.shape)
    return _canon(r)


def add32(a, b):
    with np.errstate(over="ignore", invalid="ignore"):
        return _canon(np.asarray(a, dtype=F32) + np.asarray(b, dtype=F32))


def sub32(a, b):
    with np.errstate(over="ignore", invalid="ignore"):
        return _canon(np.asarray(a, dtype=F32) - np.asarray(b, dtype=F32))


def mul32(a, b):
    with np.errstate(over="ignore", invalid="ignore"):
        return _canon(np.asarray(a, dtype=F32) * np.asarray(b, dtype=F32))


def bits(x):
    return np.asarray(x, dtype=F32).view(np.uint32)


# ---- models -----------------------------------------------------------------------------------------
def family(name):
    """('plane' | 'sphere' | 'line' | 'dense' | None, dimension)"""
    if name == "circle2":
        return "sphere", 2
    for f in ("plane", "sphere", "line", "dense"):
        if name.startswith(f) and name[len(f):].isdigit():
            return f, int(name[len(f):])
    return None, 0


def q32(name):
    """floats of a hoisted hypothesis (models.cuh model_info().Q32)"""
    fam, d = family(name)
    if fam == "plane":
        return d + 1
    if fam == "sphere":
        return d + 2
    if fam == "line":
        return 3 if d == 2 else (9 if d == 3 else 2 * d)
    if fam == "dense":
        return d + 2
    return {"line2d": 3, "absor": 12, "ray": 3, "pivot": 6, "usxw": 12, "uscp": 9}[name]


def centred(name, d):
    """models.cuh centred_component"""
    if name == "ray":
        return d < 3
    if name == "pivot":
        return d >= 9
    if name == "usxw":
        return 9 <= d < 12
    if name == "uscp":
        return False
    return family(name)[0] != "dense"


def cfg_delta(name, delta):
    """EstCfg.delta (lsqr_set_estimator): |delta| where the reference squares it"""
    fam, _ = family(name)
    return float(delta) if fam in ("sphere", "dense") or name == "pivot" else abs(float(delta))


def shifted(name):
    """Eval<M>::kShifted: counted through the carry chain"""
    return family(name)[0] in ("plane", "sphere", "dense")


def abs_form(name):
    """Eval<M>::kHasAbsForm and not shifted: the 2-D lines"""
    return name in ("line2d", "line2")


# ---- the centre and the fp32 copy ---------------------------------------------------------------------
CENTER_SAMPLE = 16384


def center_single(name, data):
    """center_sample_kernel: mean of the first min(n, 16384) records per centred component; 1024 threads sum strided records
    in order, lanes reduce by an xor butterfly, warp 0..31 totals are added in order, then one division."""
    data = np.asarray(data, dtype=np.float64)
    D = data.shape[1]
    count = min(len(data), CENTER_SAMPLE)
    c = np.zeros(20)
    if count == 0:
        return c
    rows = -(-count // 1024) * 1024
    x = np.zeros((rows, D))
    x[:count] = data[:count]
    acc = np.zeros((1024, D))
    with np.errstate(invalid="ignore", over="ignore"):
        for j in range(rows // 1024):
            acc = acc + x[j * 1024:(j + 1) * 1024]
        v = acc.reshape(32, 32, D)
        lane = np.arange(32)
        for o in (16, 8, 4, 2, 1):
            v = v + v[:, lane ^ o]
        for d in range(D):
            if not centred(name, d):
                continue
            m = 0.0
            for w in range(32):
                m += v[w, 0, d]
            m /= count
            c[d] = 0.0 if (m != m or abs(m) > 1e300) else m
    return c


def center_batch(name, data):
    """the batched kernels: the problem's first record, centred components only"""
    c = np.zeros(20)
    if len(data):
        for d in range(data.shape[1]):
            if centred(name, d):
                c[d] = data[0, d]
    return c


def copy32(name, data, c):
    """[D][n] fp32 rows: (float)(x - c); the calibrated pointer keeps t2 - p in rows 9..11 and zeros in 14..16 (ingest_kernel)"""
    data = np.asarray(data, dtype=np.float64)
    with np.errstate(invalid="ignore", over="ignore"):
        rows = [_f32(data[:, d] - c[d]) for d in range(data.shape[1])]
        if name == "uscp":
            for d in range(9, 12):
                rows[d] = _f32(data[:, d] - data[:, d + 5])
            for d in range(14, 17):
                rows[d] = np.zeros(len(data), dtype=F32)
    return rows


# ---- hoist32<M> -----------------------------------------------------------------------------------
def _quat_to_rot(s, qx, qy, qz):
    return [1 - 2 * (qy * qy + qz * qz), 2 * (qx * qy - s * qz), 2 * (qx * qz + s * qy),
            2 * (qx * qy + s * qz), 1 - 2 * (qx * qx + qz * qz), 2 * (qy * qz - s * qx),
            2 * (qx * qz - s * qy), 2 * (qy * qz + s * qx), 1 - 2 * (qx * qx + qy * qy)]


def _neg_window(wf):
    """2^32 - bits(window), stored as a float; 0 (nothing agrees) unless the window is positive"""
    return np.uint32(((1 << 32) - int(bits(wf))) if wf > 0 else 0).view(F32)


def hoist_sphere_constants(r, dl):
    """(chain start, window) of hoist_sphere in fp64: |d - r| < dl  <=>  0 <= d^2 + start < window"""
    start, width = 0.0, 0.0
    if dl > 0:
        if r >= dl:
            start, width = -(r - dl) * (r - dl), 4.0 * r * dl
        elif r + dl > 0:
            width = (r + dl) * (r + dl)
    return start, width


def hoist(name, prm, c, delta):
    """hoist32<M>(prm, c, cfg) -> Q32 fp32 constants; delta is EstCfg.delta.  A parameter vector whose first entry is NaN is
    hoist32_kernel's degenerate row: NaN constants and an empty window."""
    p = [np.float64(v) for v in prm]
    c = [np.float64(v) for v in c]
    delta = np.float64(delta)
    fam, dim = family(name)
    Q = q32(name)
    with np.errstate(invalid="ignore", over="ignore", divide="ignore"):
        if p[0] != p[0]:
            q = [CNAN] * Q
            if fam == "sphere":
                q[dim + 1] = F32(0.0)
            return q
        q = [None] * Q
        if name == "plane3":
            q[:3] = [_f32(p[0]), _f32(p[1]), _f32(p[2])]
            q[3] = _f32(delta - (p[0] * (p[3] - c[0]) + p[1] * (p[4] - c[1]) + p[2] * (p[5] - c[2])))
        elif fam == "plane":
            s = 0.0
            for i in range(dim):
                q[i] = _f32(p[i])
                s += p[i] * (p[dim + i] - c[i])
            q[dim] = _f32(delta - s)
        elif name == "line2d":
            q[:2] = [_f32(p[0]), _f32(p[1])]
            q[2] = _f32(-(p[0] * (p[2] - c[0]) + p[1] * (p[3] - c[1])))
        elif name == "line2":
            inv = 1.0 / np.sqrt(p[0] * p[0] + p[1] * p[1])
            px, py = -p[1] * inv, p[0] * inv
            q[:2] = [_f32(px), _f32(py)]
            q[2] = _f32(-(px * (p[2] - c[0]) + py * (p[3] - c[1])))
        elif name == "line3":
            inv = 1.0 / np.sqrt(p[0] * p[0] + p[1] * p[1] + p[2] * p[2])
            n = [p[0] * inv, p[1] * inv, p[2] * inv]
            a = [p[3] - c[0], p[4] - c[1], p[5] - c[2]]
            for i in range(3):
                j, k = (i + 1) % 3, (i + 2) % 3
                q[3 * i], q[3 * i + 1], q[3 * i + 2] = _f32(n[k]), _f32(-n[j]), _f32(-(a[j] * n[k] - a[k] * n[j]))
        elif fam == "line":
            for i in range(dim):
                q[i], q[dim + i] = _f32(p[i]), _f32(p[dim + i] - c[i])
        elif fam == "sphere":
            for i in range(dim):
                q[i] = _f32(p[i] - c[i])
            start, width = hoist_sphere_constants(p[dim], delta)
            q[dim] = _f32(start)
            q[dim + 1] = _neg_window(_f32(width))
        elif name == "absor":
            R = _quat_to_rot(p[0], p[1], p[2], p[3])
            q[:9] = [_f32(v) for v in R]
            for i in range(3):
                q[9 + i] = _f32(R[3 * i] * c[0] + R[3 * i + 1] * c[1] + R[3 * i + 2] * c[2] + p[4 + i] - c[3 + i])
        elif name == "ray":
            q = [_f32(p[i] - c[i]) for i in range(3)]
        elif name == "pivot":   # a negative delta admits nothing: NaN constants
            q = [_f32(p[i]) for i in range(3)] + [_f32(-(p[3 + i] - c[9 + i])) for i in range(3)]
            if delta < 0:
                q = [CNAN] * 6
        elif fam == "dense":
            q = [_f32(p[i]) for i in range(dim)] + [F32(-1.0), _f32(delta)]
        elif name == "usxw":
            q = [_f32(p[11 + i]) for i in range(6)] + [_f32(p[3 + i]) for i in range(3)] + [_f32(-(p[i] - c[9 + i])) for i in range(3)]
        elif name == "uscp":
            q = [_f32(p[8 + i]) for i in range(6)] + [_f32(p[i]) for i in range(3)]
        else:
            raise AssertionError(name)
    return [F32(v) for v in q]


# ---- Eval<M> ------------------------------------------------------------------------------------
def dist(name, q, x):
    """Eval<M>::dist: the (shifted) residual of the planes, dense systems, hyperspheres and 2-D lines"""
    fam, dim = family(name)
    if name == "plane3":
        return fma32(q[0], x[0], fma32(q[1], x[1], fma32(q[2], x[2], q[3])))
    if fam == "plane":
        s = q[dim]
        for i in range(dim - 1, -1, -1):
            s = fma32(q[i], x[i], s)
        return s
    if name in ("line2d", "line2"):
        return fma32(q[0], x[0], fma32(q[1], x[1], q[2]))
    if fam == "sphere":
        t = q[dim]
        for i in range(dim):
            w = sub32(x[i], q[i])
            t = fma32(w, w, t)
        return t
    if fam == "dense":
        s = fma32(q[dim], x[dim], q[dim + 1])
        for i in range(dim - 1, -1, -1):
            s = fma32(q[i], x[i], s)
        return s
    raise AssertionError(name)


def signed(name, q, x, fdelta, nd2):
    """Eval<M>::signed_: g with inlier <=> sign bit of g (nd2 = -(float)delta^2)"""
    fam, dim = family(name)
    if fam in ("plane", "dense"):
        s = sub32(dist(name, q, x), fdelta)
        return fma32(s, s, nd2)
    if name in ("line2d", "line2"):
        s = dist(name, q, x)
        return fma32(s, s, nd2)
    if name == "line3":
        g = nd2
        for i in range(3):
            w = fma32(x[(i + 1) % 3], q[3 * i], fma32(x[(i + 2) % 3], q[3 * i + 1], q[3 * i + 2]))
            g = fma32(w, w, g)
        return g
    if fam == "line":
        v = [sub32(x[i], q[dim + i]) for i in range(dim)]
        vn = mul32(v[0], q[0])
        for i in range(1, dim):
            vn = fma32(v[i], q[i], vn)
        nvn = sub32(F32(0.0), vn)
        g = nd2
        for i in range(dim):
            w = fma32(nvn, q[i], v[i])
            g = fma32(w, w, g)
        return g
    if name == "absor":
        g = nd2
        for i in range(3):
            d = sub32(fma32(q[3 * i], x[0], fma32(q[3 * i + 1], x[1], fma32(q[3 * i + 2], x[2], q[9 + i]))), x[3 + i])
            g = fma32(d, d, g)
        return g
    if name == "ray":
        vx, vy, vz = sub32(q[0], x[0]), sub32(q[1], x[1]), sub32(q[2], x[2])
        tt = fma32(x[3], vx, fma32(x[4], vy, mul32(x[5], vz)))
        ntt = sub32(F32(0.0), tt)
        dx, dy, dz = fma32(ntt, x[3], vx), fma32(ntt, x[4], vy), fma32(ntt, x[5], vz)
        g = fma32(dx, dx, fma32(dy, dy, fma32(dz, dz, nd2)))
        # t >= 0 && dist^2 < delta^2: both sign bits (a NaN, canonical and positive, on either side is an outlier)
        return (bits(g) & bits(ntt)).view(F32)
    if name == "pivot":
        g = nd2
        for i in range(3):
            d = add32(fma32(q[0], x[3 * i], fma32(q[1], x[3 * i + 1], fma32(q[2], x[3 * i + 2], q[3 + i]))), x[9 + i])
            g = fma32(d, d, g)
        return g
    if name in ("usxw", "uscp"):
        w = [fma32(x[12], q[k], fma32(x[13], q[3 + k], q[6 + k])) for k in range(3)]
        g = nd2
        for r in range(3):
            last = fma32(x[3 * r + 2], w[2], q[9 + r]) if name == "usxw" else mul32(x[3 * r + 2], w[2])
            e = add32(fma32(x[3 * r], w[0], fma32(x[3 * r + 1], w[1], last)), x[9 + r])
            g = fma32(e, e, g)
        return g
    raise AssertionError(name)


def decisions(name, q, x, delta, delta2, mixed):
    """fp32 decision of every datum of the fp32 rows x for the hoisted hypothesis q.  delta: EstCfg.delta, delta2: EstCfg.delta2.
    mixed: the single-problem kernels' 2-D line count -- datum i is tested as |s| < delta iff ((i >> 1) & 2) == 0 and through the
    sign of s^2 - delta^2 otherwise; the batched kernels (mixed=False) test every datum as |s| < delta."""
    fdelta = F32(delta) if delta > 0 else F32(0.0)    # fp32_delta: a threshold that is not positive admits nothing
    nd2 = F32(-F32(delta2))
    n = len(x[0])
    if shifted(name):
        fam, dim = family(name)
        if fam == "sphere":
            negk = int(bits(q[dim + 1]))
            window = ((1 << 32) - negk) & 0xFFFFFFFF
        else:
            window = int(bits(F32(2.0) * fdelta))
        if window == 0 or (fam == "sphere" and negk == 0):
            return np.zeros(n, dtype=bool)
        return bits(dist(name, q, x)).astype(np.uint64) < np.uint64(window)
    if abs_form(name):
        s = dist(name, q, x)
        with np.errstate(invalid="ignore"):
            a = np.abs(s) < fdelta
        if not mixed:
            return a
        sg = (bits(fma32(s, s, nd2)) >> np.uint32(31)).astype(bool)
        i = np.arange(n)
        return np.where(((i >> 1) & 2) == 0, a, sg)
    return (bits(signed(name, q, x, fdelta, nd2)) >> np.uint32(31)).astype(bool)


def counts(name, params, data, delta, centre="single", mixed=None):
    """fp32 count of every parameter row on data (records [n][D]).  centre: 'single' (lsqr_score) or 'batch' (the batched
    kernels); delta is what the engine was given."""
    data = np.asarray(data, dtype=np.float64)
    c = center_single(name, data) if centre == "single" else center_batch(name, data)
    x = copy32(name, data, c)
    dl = cfg_delta(name, delta)
    d2 = float(delta) * float(delta)
    mixed = (centre == "single") if mixed is None else mixed
    out = np.zeros(len(params), dtype=np.int64)
    for h, prm in enumerate(np.atleast_2d(params)):
        out[h] = int(decisions(name, hoist(name, prm, c, dl), x, dl, d2, mixed).sum())
    return out


# ---- the batched kernels' round loop ------------------------------------------------------------------
def replay(counts, valid, n, k, prob, max_tries):
    """batch_kernel's round loop (rounds of 32, strict > on the key, the stop rule after a raise).  Returns (winner, count,
    conclusive): conclusive is False when a stop-rule value t + 0.5 lies within a few ulps of an integer, where the device's
    log / pow may round to the other side."""
    tries = min(math.comb(n, k), 0xFFFFFFFF) if n >= k else 0
    tries = min(tries, max_tries)
    best, done, conclusive = 0, 0, True
    log1mp = math.log(1.0 - prob)
    while done < tries:
        keys = [(int(counts[h]) << 32) | (0xFFFFFFFF - h) if valid[h] else 0 for h in range(done, min(done + 32, tries))]
        rb = max(keys, default=0)
        if rb > best:
            best = rb
            c = best >> 32
            if c == n:
                tries = 0
            elif 0.0 < prob < 1.0 and c > 0:
                t = log1mp / math.log(1.0 - (c / n) ** k) + 0.5
                if abs(t - round(t)) <= 8 * math.ulp(t):
                    conclusive = False
                nt = 0xFFFFFFFF if t >= 4294967295.0 else int(t)
                tries = min(nt, tries)
        done += 32
    return 0xFFFFFFFF - (best & 0xFFFFFFFF), best >> 32, conclusive


# ---- the fp32 band and the float64 residuals ------------------------------------------------------------
def _quat_matrix(s, qx, qy, qz):
    return np.array(_quat_to_rot(s, qx, qy, qz)).reshape(3, 3)


def fp32_band(name, data, prm, delta):
    """Half-width (in residual units) of the band around the threshold inside which an fp32 decision may legitimately differ
    from the fp64 one: relative to the magnitude of the terms that are summed to form the residual (data in fp32 after
    centring, fused multiply-adds in fp32).  The constants are MEASURED: tools/measure_fp32_band.py finds, for the 256
    hypotheses with the largest fp32/fp64 count difference among 20 000 per estimator on 200 000 data, the distance to the
    threshold of the farthest datum that was decided differently (profiles/r02_fp32_band.jsonl); the widest needs 0.29 of this
    band, the 3-D plane 0.06 (2.8e-5 absolute for coordinates of +-1000, i.e. 1.6e-8 of the coordinate scale)."""
    if name == "usxw":                 # the summed terms: pixel * scaled rotation column, t3, t2, t1
        scale = np.abs(data[:, 12:]).max() * np.abs(prm[11:17]).max() * 2 + np.abs(prm[:6]).max() * 2 + np.abs(data[:, 9:12]).max() + 1.0
        return 4e-7 * scale
    if name == "uscp":
        scale = np.abs(data[:, 12:14]).max() * np.abs(prm[8:14]).max() * 2 + np.abs(prm[:3]).max() + np.abs(data[:, 9:12]).max() + np.abs(data[:, 14:]).max() + 1.0
        return 4e-7 * scale
    fam, dim = family(name)
    if fam == "dense":   # the summed terms are the products a_i x_i and b
        nc = data.shape[1] - 1
        scale = np.abs(data[:, :nc]).max() * np.abs(prm).max() * nc + np.abs(data[:, nc]).max() + 1.0
        return 1e-7 * scale
    scale = np.abs(data).max() + np.abs(prm).max() + 1.0
    # (the constants were measured in up to four dimensions; a residual of d terms accumulates ~sqrt(d) as much rounding)
    return 1e-7 * scale * (4.0 if (name in ("absor", "pivot", "ray") or fam == "line") else 2.0) * max(1.0, (dim / 4.0) ** 0.5)


def residual64(name, prm, data, delta):
    """|residual| in float64 numpy, and the threshold it is compared with (distance units)."""
    p = np.asarray(prm)
    fam, _ = family(name)
    if fam == "plane":
        d = data.shape[1]
        return np.abs((data - p[d:]) @ p[:d]), delta
    if name == "line2d":
        return np.abs((data - p[2:4]) @ p[0:2]), delta
    if fam == "line":
        d = data.shape[1]
        v = data - p[d:]
        w = v - (v @ p[:d])[:, None] * p[:d]
        return np.linalg.norm(w, axis=1), delta
    if fam == "sphere":
        d = data.shape[1]
        return np.abs(np.linalg.norm(data - p[:d], axis=1) - p[d]), delta
    if name == "absor":
        R = _quat_matrix(*p[:4])
        return np.linalg.norm(data[:, :3] @ R.T + p[4:7] - data[:, 3:], axis=1), delta
    if name == "ray":
        v = p[:3] - data[:, :3]
        t = np.sum(v * data[:, 3:], axis=1)
        r = np.linalg.norm(v - t[:, None] * data[:, 3:], axis=1)
        r[t < 0] = np.inf
        return r, delta
    if name == "pivot":
        R = data[:, :9].reshape(-1, 3, 3)
        return np.linalg.norm(np.einsum("nij,j->ni", R, p[:3]) + data[:, 9:] - p[3:6], axis=1), delta
    if fam == "dense":
        nc = data.shape[1] - 1
        return np.abs(data[:, :nc] @ p[:nc] - data[:, nc]), delta
    if name == "usxw":
        R2 = data[:, :9].reshape(-1, 3, 3)
        w = np.outer(data[:, 12], p[11:14]) + np.outer(data[:, 13], p[14:17]) + p[3:6]
        return np.linalg.norm(np.einsum("nij,nj->ni", R2, w) + data[:, 9:12] - p[0:3], axis=1), delta
    if name == "uscp":
        R2 = data[:, :9].reshape(-1, 3, 3)
        w = np.outer(data[:, 12], p[8:11]) + np.outer(data[:, 13], p[11:14]) + p[0:3]
        return np.linalg.norm(np.einsum("nij,nj->ni", R2, w) + data[:, 9:12] - data[:, 14:17], axis=1), delta
    raise AssertionError(name)


NAMES = sorted(MODELS, key=MODELS.get)
assert len(NAMES) == 34 and all(INFO[MODELS[n]][0] > 0 for n in NAMES)
