"""ORACLE (test infrastructure, not product code) -- first hits of rays on a 3D triangle mesh.

An engine extension with no counterpart in the reference: `raycast` below is the DEFINITION that ctr_mt3d_raycast is
tested against, parity UNPINNED by the reference, like oracle/mt3d_closest.py.  It is a pure function of a mesh (as the
engine's fetch returns it), the rays and a t range.  Every operation is one separately rounded fp64 operation in a
fixed order, so the device result equals it bit for bit.
"""
import numpy as np

PAD = 2.0 ** -40                      # the leaf box pad of ctr_mt3d_closest's k_cq_box, relative to max|coordinate|


def ray_setup(O, D):
    """(kx, ky, kz, Sx, Sy, Sz) per ray (arrays [R]): step 1 of the definition.  kz = the first index of the largest
    |d_k|; kx = (kz+1) % 3, ky = (kx+1) % 3, swapped when d[kz] < 0; Sx = d[kx]/d[kz], Sy = d[ky]/d[kz], Sz = 1/d[kz]."""
    D = np.asarray(D, np.float64)
    kz = np.argmax(np.abs(D), axis=1)                                   # argmax: the first on a tie
    kx = (kz + 1) % 3
    ky = (kx + 1) % 3
    r = np.arange(len(D))
    dz = D[r, kz]
    neg = dz < 0
    kx, ky = np.where(neg, ky, kx), np.where(neg, kx, ky)
    with np.errstate(divide="ignore", over="ignore", invalid="ignore"):
        return kx, ky, kz, D[r, kx] / dz, D[r, ky] / dz, 1.0 / dz


def triangle_hits(O, D, a, b, c, t_min, t_max):
    """The watertight test of the definition for ray i against triangle i (arrays [n, 3] fp64, t_min / t_max scalars
    or [n]).  Returns (hit [n] bool, t, U, V, W, det, point [n, 3]); values where hit is False are meaningless."""
    n = len(O)
    r = np.arange(n)
    kx, ky, kz, Sx, Sy, Sz = ray_setup(O, D)
    with np.errstate(divide="ignore", over="ignore", invalid="ignore", under="ignore"):
        def shear(v):
            A = v - O                                                    # step 2: shift ...
            az = A[r, kz]
            return A[r, kx] - Sx * az, A[r, ky] - Sy * az, az           # ... and shear
        Ax, Ay, Az = shear(a)
        Bx, By, Bz = shear(b)
        Cx, Cy, Cz = shear(c)
        U = Cx * By - Cy * Bx                                            # step 3: the edge functions
        V = Ax * Cy - Ay * Cx
        W = Bx * Ay - By * Ax
        miss = ((U < 0) | (V < 0) | (W < 0)) & ((U > 0) | (V > 0) | (W > 0))     # step 4
        det = (U + V) + W
        miss |= det == 0
        T = (U * (Sz * Az) + V * (Sz * Bz)) + W * (Sz * Cz)            # step 5
        t = T / det
        P = O + t[:, None] * D                                           # step 6: multiply, then add, per axis
        lo = np.minimum(np.minimum(a, b), c)                             # step 7: the padded box
        hi = np.maximum(np.maximum(a, b), c)
        m = np.maximum(np.abs(lo), np.abs(hi)).max(axis=1)
        pad = (m * PAD)[:, None]
        inbox = ((lo - pad <= P) & (P <= hi + pad)).all(axis=1)
        hit = ~miss & (t_min <= t) & (t <= t_max) & inbox
    return hit, t, U, V, W, det, P


def _rays(origins, directions, t_min, t_max):
    O = np.asarray(origins).astype(np.float64).reshape(-1, 3)
    D = np.asarray(directions).astype(np.float64).reshape(-1, 3)
    if O.shape != D.shape:
        raise ValueError("origins and directions must have the same shape")
    t_min, t_max = float(t_min), float(t_max)
    if np.isnan(t_min) or np.isnan(t_max) or not t_min <= t_max:
        raise ValueError("t_min and t_max must not be NaN, and t_min <= t_max")
    if not (np.isfinite(O).all() and np.isfinite(D).all()):
        raise ValueError("ray origins and directions must be finite")
    if len(D) and not (D != 0).any(axis=1).all():
        raise ValueError("ray directions must not be zero")
    return O, D, t_min, t_max


def raycast(verts, tris, origins, directions, t_min=0.0, t_max=np.inf, prune=False, chunk=1 << 19):
    """(dict(t [R] f64, triangle [R] int32, weights [R, 3] f64, point [R, 3] f64, side [R] int8), n_hit) --
    ctr_mt3d_raycast's definition.

    Positions (fp32 or fp64 geometry), origins and directions (fp32 or fp64) are widened to fp64; every operation
    below is one fp64 operation, rounded on its own (no fused multiply-add), in the order written.  For ray (o, d) and
    triangle (a, b, c), corners in stored order, Woop, Benthin and Wald's watertight test (JCGT 2(1), 2013):
      1. kz = the index of the largest |d_k| (the first on a tie), kx = (kz+1) % 3, ky = (kx+1) % 3; kx and ky swapped
         when d[kz] < 0.  Sx = d[kx]/d[kz], Sy = d[ky]/d[kz], Sz = 1/d[kz].
      2. A = a - o, Ax = A[kx] - Sx*A[kz], Ay = A[ky] - Sy*A[kz]; the same for B and C.
      3. U = Cx*By - Cy*Bx, V = Ax*Cy - Ay*Cx, W = Bx*Ay - By*Ax.
      4. A miss when (U<0 or V<0 or W<0) and (U>0 or V>0 or W>0).  det = (U+V)+W; a miss when det == 0.
      5. T = (U*(Sz*A[kz]) + V*(Sz*B[kz])) + W*(Sz*C[kz]), t = T/det.
      6. p = o + t*d per axis (multiply, then add).
      7. A hit when t_min <= t <= t_max and p lies in the triangle's padded box [min - pad, max + pad] per axis, with
         pad = 2^-40 max|coordinate of a, b, c| (the box k_cq_box computes in fp64 before rounding outward to fp32).
      8. weights = (U/det, V/det, W/det), of a, b and c; side = +1 when det > 0, else -1.  det > 0 means
         dot(d, cross(b-a, c-a)) < 0: the ray arrives from the side the triangle faces.  On the raw mesh, whose
         triangles face the high side of the field, +1 means the origin is on the high side.
      9. The winner of a ray is the hit with the smallest t, the smallest triangle index on a tie.  A ray with no hit
         gets t = +inf, triangle -1, weights and point NaN and side 0.  n_hit counts the rays with a hit.
    Watertightness follows from steps 2 and 3: the two triangles on an edge compute that edge's function from the same
    transformed corners, so the values are exact negatives of each other (or both zero), and a ray through an edge or
    a vertex cannot pass between the triangles around it.
    The box guard of step 7 rejects only hits whose t is rounding noise: a grazing ray, or a sliver whose det is the
    rounding error of its edge functions, can give a t that puts p far from the triangle.  Any other computed p lies
    within a few rounding errors of the triangle, far inside the pad.  The guard also makes pruning provable: every
    accepted p lies in its triangle's outward-rounded fp32 leaf box, and so in the box of every ancestor in a tree over
    those boxes, so a traversal that never skips a box holding a computed p with t in [t_min, best] finds what brute
    force finds (DESIGN.md, "Ray casting").

    Brute force over every triangle, in chunks.  prune=True evaluates only the triangles whose padded box a
    conservative slab test admits: the boxes widened by 1e-9 (max|corner| + |o|) per axis (far above the rounding of
    p) and the slab ends by 1e-12 relative, through two levels of blocks of 64 triangles in Morton order.  The result
    is the same (tests/test_oracle_raycast_cpu.py checks it against brute force)."""
    V = np.asarray(verts).astype(np.float64).reshape(-1, 3)
    T = np.asarray(tris, np.int64).reshape(-1, 3)
    O, D, t_min, t_max = _rays(origins, directions, t_min, t_max)
    if len(T) and (T.min() < 0 or T.max() >= len(V)):
        raise ValueError("triangle ids outside [0, n_verts)")
    nR, nT = len(O), len(T)
    best_t = np.full(nR, np.inf)
    best_i = np.full(nR, -1, np.int64)
    if nR and nT:
        if prune:
            ri, ti = _candidates(V, T, O, D, t_min, t_max)
        else:
            ri = ti = None
        _reduce(V, T, O, D, t_min, t_max, ri, ti, best_t, best_i, chunk)
    found = best_i >= 0
    out = dict(t=np.where(found, best_t, np.inf), triangle=np.where(found, best_i, -1).astype(np.int32),
               weights=np.full((nR, 3), np.nan), point=np.full((nR, 3), np.nan), side=np.zeros(nR, np.int8))
    if found.any():
        r = np.nonzero(found)[0]
        t3 = T[best_i[r]]
        hit, t, U, Vv, W, det, P = triangle_hits(O[r], D[r], V[t3[:, 0]], V[t3[:, 1]], V[t3[:, 2]], t_min, t_max)
        assert hit.all() and np.array_equal(t, best_t[r])
        with np.errstate(divide="ignore", invalid="ignore"):
            out["weights"][r] = np.stack([U / det, Vv / det, W / det], axis=1)
        out["point"][r] = P
        out["side"][r] = np.where(det > 0, 1, -1)
        out["t"][r] = t
    return out, int(found.sum())


def _reduce(V, T, O, D, t_min, t_max, ri, ti, best_t, best_i, chunk):
    "the smallest (t, triangle) hit per ray over the pairs (ri, ti), or over every pair when ri is None"
    nR, nT = len(O), len(T)
    if ri is None:
        step_r = max(1, chunk // nT)
        step_t = min(nT, chunk)
        pieces = ((np.repeat(np.arange(r0, min(nR, r0 + step_r)), min(nT, t0 + step_t) - t0),
                   np.tile(np.arange(t0, min(nT, t0 + step_t)), min(nR, r0 + step_r) - r0))
                  for r0 in range(0, nR, step_r) for t0 in range(0, nT, step_t))
    else:
        pieces = ((ri[s:s + chunk], ti[s:s + chunk]) for s in range(0, len(ri), chunk))
    for pr, pt in pieces:
        t3 = T[pt]
        hit, t, *_ = triangle_hits(O[pr], D[pr], V[t3[:, 0]], V[t3[:, 1]], V[t3[:, 2]], t_min, t_max)
        pr, pt, t = pr[hit], pt[hit], t[hit]
        if not len(pr):
            continue
        o = np.lexsort((pt, t, pr))                                      # by ray, then t, then triangle
        first = o[np.r_[True, pr[o][1:] != pr[o][:-1]]]
        r, tt, ii = pr[first], t[first], pt[first]
        better = (tt < best_t[r]) | ((tt == best_t[r]) & (ii < best_i[r])) | (best_i[r] < 0)
        best_t[r[better]] = tt[better]
        best_i[r[better]] = ii[better]


def _slab(O, D, lo, hi, t_min, t_max):
    "conservative: False only when no p = o + t d (computed) with t in [t_min, t_max] lies in the box (lo, hi)"
    with np.errstate(divide="ignore", over="ignore", invalid="ignore", under="ignore"):
        eps = 1e-9 * (np.maximum(np.abs(lo), np.abs(hi)).max(axis=-1, keepdims=True) + np.abs(O)) + 1e-300
        lo, hi = lo - eps, hi + eps
        zero = D == 0
        t1, t2 = (lo - O) / D, (hi - O) / D
        tn = np.nan_to_num(np.minimum(t1, t2), nan=-np.inf, posinf=np.finfo(np.float64).max)
        tf = np.nan_to_num(np.maximum(t1, t2), nan=np.inf, neginf=-np.finfo(np.float64).max)
        tn = np.where(zero, np.where((lo <= O) & (O <= hi), -np.inf, np.inf), tn - 1e-12 * np.abs(tn) - 1e-300)
        tf = np.where(zero, np.where((lo <= O) & (O <= hi), np.inf, -np.inf), tf + 1e-12 * np.abs(tf) + 1e-300)
        return np.maximum(tn.max(axis=-1), t_min) <= np.minimum(tf.min(axis=-1), t_max)


def _candidates(V, T, O, D, t_min, t_max, block=64, rays_per_piece=256):
    "(ray, triangle) pairs whose padded box the slab test admits, through two levels of blocks in Morton order"
    a, b, c = V[T[:, 0]], V[T[:, 1]], V[T[:, 2]]
    lo = np.minimum(np.minimum(a, b), c)
    hi = np.maximum(np.maximum(a, b), c)
    pad = (np.maximum(np.abs(lo), np.abs(hi)).max(axis=1) * PAD)[:, None]
    lo, hi = lo - pad, hi + pad
    cen = (lo + hi) / 2
    s_lo, s_hi = cen.min(axis=0), cen.max(axis=0)
    q = np.clip(((cen - s_lo) / np.maximum(s_hi - s_lo, 1e-300) * 1023).astype(np.int64), 0, 1023)
    code = np.zeros(len(T), np.int64)
    for bit in range(10):
        for k in range(3):
            code |= ((q[:, k] >> bit) & 1) << (3 * bit + 2 - k)
    order = np.argsort(code, kind="stable")
    lo, hi = lo[order], hi[order]
    levels = [(lo, hi)]
    while len(levels[-1][0]) > block:
        l, h = levels[-1]
        nb = -(-len(l) // block)
        fill = nb * block - len(l)
        l = np.concatenate([l, np.full((fill, 3), np.inf)]).reshape(nb, block, 3).min(axis=1)
        h = np.concatenate([h, np.full((fill, 3), -np.inf)]).reshape(nb, block, 3).max(axis=1)
        levels.append((l, h))
    out_r, out_t = [], []
    for r0 in range(0, len(O), rays_per_piece):
        r = np.arange(r0, min(len(O), r0 + rays_per_piece))
        l, h = levels[-1]
        pr = np.repeat(r, len(l))
        pn = np.tile(np.arange(len(l)), len(r))
        keep = _slab(O[pr], D[pr], l[pn], h[pn], t_min, t_max)
        pr, pn = pr[keep], pn[keep]
        for lev in range(len(levels) - 2, -1, -1):
            l, h = levels[lev]
            pr = np.repeat(pr, block)
            pn = (pn[:, None] * block + np.arange(block)).reshape(-1)
            ok = pn < len(l)
            pr, pn = pr[ok], pn[ok]
            keep = np.zeros(len(pr), bool)
            for s in range(0, len(pr), 1 << 20):
                sl = slice(s, s + (1 << 20))
                keep[sl] = _slab(O[pr[sl]], D[pr[sl]], l[pn[sl]], h[pn[sl]], t_min, t_max)
            pr, pn = pr[keep], pn[keep]
        out_r.append(pr)
        out_t.append(order[pn])
    return np.concatenate(out_r), np.concatenate(out_t)
