"""UV atlas of the mesh exporter (host, init-time, numpy + scipy).

threestudio's `mesh-exporter` unwraps with xatlas; this atlas is the project's own, deterministic and overlap-free by
construction, then verified:

  1. classes: each face gets the dominant axis and sign of its geometric normal (6 classes);
  2. charts: connected components of same-class faces sharing an undirected edge;
  3. projection: orthographic along the class axis, one coordinate mirrored for negative classes, so every projected
     triangle is counter-clockwise.  This stretches lengths by up to sqrt(3); it is not xatlas's distortion-driven unwrap;
  4. one global texel density `s` (texels per unit length) for every chart, chart boxes shelf-packed with a gutter of
     2 * padding + 1 texels (and `padding` texels to the border), `s` shrunk by a fixed factor until everything fits;
  5. every chart vertex snapped to fixed point with 8 sub-texel bits: the integers are what the rasteriser reads;
  6. every face rasterised with the same integer rule as dm_uv_raster; a chart that covers a texel centre twice is a
     folded projection (e.g. a helicoid) and is split into one chart per face, then everything is packed again.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np
import scipy.sparse as sp
from scipy.sparse.csgraph import connected_components

SUBPIX = 256          # 8 sub-texel bits
SHRINK = 0.9          # density factor per failed packing pass
_DROP = {0: (1, 2), 1: (2, 0), 2: (0, 1)}   # cyclic order: the projected signed area equals the normal's component


@dataclass
class Atlas:
    v_tex: np.ndarray        # [Vt, 2] float32, uv in [0, 1]: u = column, v = row (row r <-> v = (r + 0.5) / T)
    t_tex_idx: np.ndarray    # [F, 3] int32 into v_tex
    uv_fixed: np.ndarray     # [Vt, 2] int32 texel coordinates * 256 (what the rasteriser reads)
    face_chart: np.ndarray   # [F] int64 chart id of every face
    density: float           # s, texels per unit length
    texture_size: int
    padding: int


def face_classes(v: np.ndarray, f: np.ndarray) -> np.ndarray:
    n = np.cross(v[f[:, 1]] - v[f[:, 0]], v[f[:, 2]] - v[f[:, 0]])
    axis = np.argmax(np.abs(n), 1)
    neg = n[np.arange(len(f)), axis] < 0
    return axis * 2 + neg


def charts_of(f: np.ndarray, cls: np.ndarray) -> np.ndarray:
    """connected components of same-class faces that share an undirected edge"""
    F = len(f)
    e = np.sort(np.concatenate([f[:, [0, 1]], f[:, [1, 2]], f[:, [2, 0]]], 0), 1)
    fid = np.tile(np.arange(F), 3)
    order = np.lexsort((cls[fid], e[:, 1], e[:, 0]))
    e, fid = e[order], fid[order]
    same = (e[1:] == e[:-1]).all(1) & (cls[fid[1:]] == cls[fid[:-1]])
    a, b = fid[:-1][same], fid[1:][same]
    g = sp.coo_matrix((np.ones(len(a)), (a, b)), shape=(F, F))
    return connected_components(g, directed=False)[1].astype(np.int64)


def raster_fixed(uvf: np.ndarray, tri: np.ndarray, T: int, chunk: int = 1 << 22):
    """Covered texel centres of every face, dm_uv_raster's integer rule -> (texel ids r*T+c, face ids).  Chunked over
    faces so that the candidate lists stay bounded."""
    P = uvf.astype(np.int64)[tri]
    x, y = P[..., 0], P[..., 1]
    area = (x[:, 1] - x[:, 0]) * (y[:, 2] - y[:, 0]) - (x[:, 2] - x[:, 0]) * (y[:, 1] - y[:, 0])
    c_lo = np.maximum((x.min(1) - 128 + 255) // 256, 0); c_hi = np.minimum((x.max(1) - 128) // 256, T - 1)
    r_lo = np.maximum((y.min(1) - 128 + 255) // 256, 0); r_hi = np.minimum((y.max(1) - 128) // 256, T - 1)
    nw, nh = c_hi - c_lo + 1, r_hi - r_lo + 1
    cnt = np.where((area > 0) & (nw > 0) & (nh > 0), nw * nh, 0)
    cum = np.cumsum(cnt)
    texels, faces = [], []
    start = 0
    while start < len(tri):
        base = cum[start - 1] if start else 0
        stop = max(int(np.searchsorted(cum, base + chunk, "right")), start + 1)
        fs = np.arange(start, stop)
        fid = np.repeat(fs, cnt[fs])
        if len(fid):
            k = np.arange(len(fid)) - np.repeat(cum[fs] - cnt[fs] - base, cnt[fs])
            c = c_lo[fid] + k % nw[fid]
            r = r_lo[fid] + k // nw[fid]
            px, py = 256 * c + 128, 256 * r + 128
            inside = np.ones(len(fid), bool)
            for i, j in ((0, 1), (1, 2), (2, 0)):
                ax, ay, bx, by = x[fid, i], y[fid, i], x[fid, j], y[fid, j]
                dx, dy = bx - ax, by - ay
                E = dx * (py - ay) - dy * (px - ax)
                inside &= (E > 0) | ((E == 0) & ((dy > 0) | ((dy == 0) & (dx < 0))))
            texels.append((r * T + c)[inside]); faces.append(fid[inside])
        start = stop
    if not texels:
        return np.zeros(0, np.int64), np.zeros(0, np.int64)
    return np.concatenate(texels), np.concatenate(faces)


def _project(v, f, cls):
    """[F,3,2] projected corner coordinates (counter-clockwise for every non-degenerate face)"""
    uv = np.empty((len(f), 3, 2))
    for c in range(6):
        sel = cls == c
        a, b = _DROP[c // 2]
        uv[sel, :, 0] = v[f[sel]][..., a] * (-1.0 if c % 2 else 1.0)
        uv[sel, :, 1] = v[f[sel]][..., b]
    return uv


def _pack(w, h, T, pad, s):
    """shelf packing at density s -> integer box origins [n, 2] (texels), or None if the charts do not fit"""
    gut = 2 * pad + 1
    W, H = w * s, h * s
    order = np.lexsort((np.arange(len(w)), -H))
    org = np.zeros((len(w), 2), np.int64)
    x = y = pad
    shelf = 0.0
    for i in order:
        if W[i] > T - 2 * pad:
            return None
        if x + W[i] > T - pad:
            x, y = pad, y + int(np.ceil(shelf)) + gut
            shelf = 0.0
        if y + H[i] > T - pad:
            return None
        org[i] = (x, y)
        shelf = max(shelf, H[i])
        x += int(np.ceil(W[i])) + gut
    return org


def build_atlas(v_pos, t_pos_idx, texture_size: int, padding: int = 2) -> Atlas:
    T, pad = int(texture_size), int(padding)
    if not 16 <= T <= 8192:
        raise ValueError(f"texture_size {T} outside [16, 8192]")
    if pad < 0:
        raise ValueError("padding must be >= 0")
    v = np.asarray(v_pos, np.float64)
    f = np.asarray(t_pos_idx, np.int64)
    if f.ndim != 2 or f.shape[0] == 0 or f.shape[1] != 3:
        raise ValueError("empty mesh: nothing to unwrap")
    F = len(f)
    cls = face_classes(v, f)
    proj = _project(v, f, cls)
    chart = charts_of(f, cls)
    gut = 2 * pad + 1
    while True:
        _, chart = np.unique(chart, return_inverse=True)
        n_ch = int(chart.max()) + 1
        lo = np.full((n_ch, 2), np.inf); hi = np.full((n_ch, 2), -np.inf)
        np.minimum.at(lo, chart, proj.min(1)); np.maximum.at(hi, chart, proj.max(1))
        w, h = hi[:, 0] - lo[:, 0], hi[:, 1] - lo[:, 1]
        # first guess: the boxes plus their gutters fill the usable square; then shrink until the shelves fit
        A, B, C = w @ h, gut * (w + h).sum(), n_ch * gut * gut - float(T - 2 * pad) ** 2
        if C >= 0:
            raise ValueError(f"{n_ch} charts do not fit a {T}^2 texture with padding {pad}")
        s = (-B + np.sqrt(B * B - 4 * A * C)) / (2 * A) if A > 0 else (-C / B if B > 0 else 1.0)
        org = _pack(w, h, T, pad, s)
        while org is None:
            s *= SHRINK
            if s * max(w.max(), h.max()) < 1e-3:
                raise ValueError(f"{n_ch} charts do not fit a {T}^2 texture with padding {pad}")
            org = _pack(w, h, T, pad, s)
        # one vt per (chart, vertex): faces inside a chart share corners exactly
        key = chart[:, None] * len(v) + f
        uniq, inv = np.unique(key.reshape(-1), return_inverse=True)
        t_tex = inv.reshape(F, 3)
        tex = (proj - lo[chart][:, None, :]) * s + org[chart][:, None, :]
        fixed = np.zeros((len(uniq), 2), np.int64)
        fixed[t_tex.reshape(-1)] = np.rint(tex.reshape(-1, 2) * SUBPIX).astype(np.int64)
        fixed = np.clip(fixed, SUBPIX * pad, SUBPIX * (T - pad))
        tid, fid = raster_fixed(fixed, t_tex, T)
        cnt = np.bincount(tid, minlength=T * T)
        folded = np.unique(chart[fid[cnt[tid] > 1]])
        if len(folded) == 0:
            break
        split = np.isin(chart, folded)
        chart = np.where(split, n_ch + np.arange(F), chart)
    return Atlas(v_tex=(fixed / (SUBPIX * T)).astype(np.float32), t_tex_idx=t_tex.astype(np.int32),
                 uv_fixed=fixed.astype(np.int32), face_chart=chart, density=float(s), texture_size=T, padding=pad)
