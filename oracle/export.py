"""CPU restatement of the mesh exporter's texture bake (dreammat_b200/texbake.py), used by the tests.

Integer UV raster (one face at a time, the top-left rule of dm_uv_raster), float64 interpolation, the hash grid + MLP of
`render.geometry_forward`, DreamMatMaterial.export (dreammat_material.py:765-797), the reference's uv_padding quantisation
(uint8)(x*255), and the nearest-covered-texel fill from scipy.ndimage.distance_transform_edt.
"""
import numpy as np
import torch

from . import render as O


def raster(uv_fixed, tri_uv, T):
    """-> owner [T*T] int64 (-1 = empty), bary [T*T, 3] float64, count [T*T] (centres covered per texel)"""
    uvf = np.asarray(uv_fixed, np.int64)
    owner = np.full(T * T, -1, np.int64)
    bary = np.zeros((T * T, 3))
    count = np.zeros(T * T, np.int64)
    for fi, (a, b, c) in enumerate(np.asarray(tri_uv, np.int64)):
        (x0, y0), (x1, y1), (x2, y2) = uvf[a], uvf[b], uvf[c]
        area = (x1 - x0) * (y2 - y0) - (x2 - x0) * (y1 - y0)
        if area <= 0:
            continue
        cs = np.arange(max(-((128 - min(x0, x1, x2)) // 256), 0), min((max(x0, x1, x2) - 128) // 256, T - 1) + 1)
        rs = np.arange(max(-((128 - min(y0, y1, y2)) // 256), 0), min((max(y0, y1, y2) - 128) // 256, T - 1) + 1)
        if len(cs) == 0 or len(rs) == 0:
            continue
        R, Cc = np.meshgrid(rs, cs, indexing="ij")
        px, py = 256 * Cc + 128, 256 * R + 128
        E, ok = [], np.ones(R.shape, bool)
        for (ax, ay), (bx, by) in (((x0, y0), (x1, y1)), ((x1, y1), (x2, y2)), ((x2, y2), (x0, y0))):
            dx, dy = bx - ax, by - ay
            e = dx * (py - ay) - dy * (px - ax)
            top_left = dy > 0 or (dy == 0 and dx < 0)
            ok &= (e > 0) | ((e == 0) & top_left)
            E.append(e)
        ids = (R * T + Cc)[ok]
        owner[ids] = fi
        count[ids] += 1
        bary[ids] = np.stack([E[1][ok], E[2][ok], E[0][ok]], -1) / float(area)
    return owner, bary, count


def texel_points(owner, bary, v_pos, t_pos_idx):
    """row-major covered texels -> (texel ids, points [n, 3] float64)"""
    tex = np.nonzero(owner >= 0)[0]
    v = np.asarray(v_pos, np.float64)
    f = np.asarray(t_pos_idx, np.int64)[owner[tex]]
    return tex, np.einsum("nk,nkc->nc", bary[tex], v[f])


def material_export(features, min_metallic=0.0, max_metallic=0.9, min_roughness_squre=0.01, max_roughness_squre=0.9):
    m = torch.sigmoid(torch.as_tensor(features, dtype=torch.float64))
    return torch.cat([m[:, :3], m[:, 3:4] * (max_metallic - min_metallic) + min_metallic,
                      torch.sqrt(m[:, 4:5] * (max_roughness_squre - min_roughness_squre) + min_roughness_squre + 1e-7)], -1).numpy()


def quantise(x):
    return np.floor(np.asarray(x) * 255.0).astype(np.uint8)


def bake(uv_fixed, tri_uv, T, v_pos, t_pos_idx, grid, W1, W2, material_kwargs=None):
    """-> dict(owner, bary, texels, points, maps [T*T, 5] uint8 before the fill, filled [T*T, 5] uint8, src [T*T])"""
    from scipy.ndimage import distance_transform_edt
    owner, bary, count = raster(uv_fixed, tri_uv, T)
    tex, pts = texel_points(owner, bary, v_pos, t_pos_idx)
    meta, _ = O.hashgrid_meta()
    feats = O.geometry_forward(torch.from_numpy(pts), torch.as_tensor(grid, dtype=torch.float64),
                               torch.as_tensor(W1, dtype=torch.float64), torch.as_tensor(W2, dtype=torch.float64), meta)
    q = quantise(material_export(feats, **(material_kwargs or {})))
    maps = np.zeros((T * T, 5), np.uint8)
    maps[tex] = q
    empty = (owner < 0).reshape(T, T)
    _, (ir, ic) = distance_transform_edt(empty, return_indices=True)
    src = (ir * T + ic).reshape(-1)
    return dict(owner=owner, bary=bary, count=count, texels=tex, points=pts, features=feats.numpy(), maps=maps,
                filled=maps[src], src=src)
