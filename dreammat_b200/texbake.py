"""Texture bake of the mesh exporter: trained geometry + material -> albedo / metallic / roughness maps on a UV atlas.

Stages (include/dreammat_b200.h, N5): atlas (host, uvatlas.py) -> dm_uv_raster -> dm_compact_mask -> dm_texel_positions
-> dm_hashgrid_mlp_fwd -> dm_material_export (activation + (uint8)(x*255) + scatter) -> dm_seam_fill.

Map layout: texel (r, c) is uv = ((c + 0.5) / T, (r + 0.5) / T), nvdiffrast's layout for uv_clip = v_tex * 2 - 1; row 0
is v = 0.  Departure from the reference's padding: every empty texel takes the value of a covered texel at the exact
minimal Euclidean distance instead of cv2.inpaint (Telea); covered texels are identical, hole texels differ.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass
from typing import Any, Dict, Optional

import numpy as np
import torch

from . import render_ops as R
from . import uvatlas
from ._cabi import MaterialCfg, check, lib, ptr, stream_ptr


@dataclass
class ExportedMesh:
    """the attributes threestudio's `save_obj` reads from `params["mesh"]`"""
    v_pos: torch.Tensor
    t_pos_idx: torch.Tensor
    v_nrm: Optional[torch.Tensor] = None
    v_tex: Optional[torch.Tensor] = None
    t_tex_idx: Optional[torch.Tensor] = None
    v_rgb: Optional[torch.Tensor] = None


def _check_inputs(geometry, material):
    from .system import DreamMatMaterial, DreamMatMesh
    if not isinstance(geometry, DreamMatMesh):
        raise TypeError(f"the exporter bakes dreammat_b200 geometry only, got {type(geometry).__name__}")
    if not isinstance(material, DreamMatMaterial):
        raise TypeError(f"the exporter bakes dreammat_b200 materials only, got {type(material).__name__}")


def export_cfg(material) -> MaterialCfg:
    """dm_material_cfg of DreamMatMaterial.export: the roughness fields hold the squared-roughness range"""
    c = material.cfg
    return MaterialCfg(c.min_metallic, c.max_metallic, c.min_roughness_squre, c.max_roughness_squre, 0, 0)


def _features(geometry, points):
    f = torch.empty(points.shape[0], geometry.cfg.n_feature_dims, device=points.device)
    check(lib().dm_hashgrid_mlp_fwd(C.byref(geometry.hg), ptr(points), points.shape[0], ptr(geometry.grid), ptr(geometry.W1),
                                    ptr(geometry.W2), ptr(f), stream_ptr()), "dm_hashgrid_mlp_fwd")
    return f


def vertex_material(geometry, material) -> torch.Tensor:
    """DreamMatMaterial.export at the mesh vertices -> [V, 5] (albedo rgb, metallic, roughness) on the device"""
    _check_inputs(geometry, material)
    pts = geometry.v_pos.to(geometry.device, torch.float32).contiguous()
    f = _features(geometry, pts)
    out = torch.empty(pts.shape[0], 5, device=pts.device)
    check(lib().dm_material_export(C.byref(export_cfg(material)), ptr(f), pts.shape[0], ptr(out), None, None, None, None,
                                   stream_ptr()), "dm_material_export")
    return out


def bake_textures(geometry, material, texture_size: int = 1024, padding: int = 2, atlas=None,
                  return_debug: bool = False, mark=None) -> Dict[str, Any]:
    """-> v_pos, t_pos_idx, v_tex, t_tex_idx (host), map_Kd [T,T,3], map_Pm [T,T,1], map_Pr [T,T,1] (float32 k/255,
    device).  return_debug adds the intermediate buffers (owner, bary, mask, texels, points, uint8 maps, fill source);
    mark(stage) is called after each device stage (scripts/bench_export.py records CUDA events there)."""
    mark = mark or (lambda stage: None)
    _check_inputs(geometry, material)
    if geometry.cfg.n_feature_dims != 5:
        raise ValueError("the bake reads albedo / metallic / roughness from 5 feature channels")
    T = int(texture_size)
    if atlas is None:
        atlas = uvatlas.build_atlas(geometry.v_pos.numpy(), geometry.t_pos_idx.numpy(), T, padding)
    dev = geometry.device
    st = stream_ptr()
    uvf = torch.from_numpy(atlas.uv_fixed).to(dev)
    tri_uv = torch.from_numpy(atlas.t_tex_idx).to(dev)
    v_pos = geometry.v_pos.to(dev, torch.float32).contiguous()
    t_pos = geometry.t_pos_idx.to(dev, torch.int32).contiguous()
    n_tex = T * T
    owner = torch.empty(n_tex, dtype=torch.int32, device=dev)
    bary = torch.empty(n_tex, 3, device=dev)
    mask = torch.empty(n_tex, dtype=torch.uint8, device=dev)
    mark("start")
    check(lib().dm_uv_raster(ptr(uvf), ptr(tri_uv), tri_uv.shape[0], T, ptr(owner), ptr(bary), ptr(mask), st), "dm_uv_raster")
    mark("raster")
    texels = R.compact_mask(mask)
    n = int(texels.shape[0])
    points = torch.empty(n, 3, device=dev)
    check(lib().dm_texel_positions(ptr(texels), n, ptr(owner), ptr(bary), ptr(v_pos), ptr(t_pos), ptr(points), st),
          "dm_texel_positions")
    mark("positions")
    feats = _features(geometry, points)
    mark("hashgrid")
    kd8 = torch.empty(n_tex, 3, dtype=torch.uint8, device=dev)
    pm8 = torch.empty(n_tex, dtype=torch.uint8, device=dev)
    pr8 = torch.empty(n_tex, dtype=torch.uint8, device=dev)
    check(lib().dm_material_export(C.byref(export_cfg(material)), ptr(feats), n, None, ptr(texels), ptr(kd8), ptr(pm8),
                                   ptr(pr8), st), "dm_material_export")
    mark("export")
    scratch = torch.empty(4 * n_tex, dtype=torch.int32, device=dev)
    src = torch.empty(n_tex, dtype=torch.int32, device=dev)
    kd = torch.empty(T, T, 3, device=dev)
    pm = torch.empty(T, T, 1, device=dev)
    pr = torch.empty(T, T, 1, device=dev)
    check(lib().dm_seam_fill(ptr(mask), T, ptr(kd8), ptr(pm8), ptr(pr8), ptr(scratch), ptr(src), ptr(kd), ptr(pm), ptr(pr), st),
          "dm_seam_fill")
    mark("fill")
    out = {"v_pos": geometry.v_pos, "t_pos_idx": geometry.t_pos_idx, "v_tex": torch.from_numpy(atlas.v_tex),
           "t_tex_idx": torch.from_numpy(atlas.t_tex_idx), "map_Kd": kd, "map_Pm": pm, "map_Pr": pr}
    if return_debug:
        out.update(atlas=atlas, owner=owner, bary=bary, mask=mask, texels=texels, points=points, features=feats,
                   kd8=kd8, pm8=pm8, pr8=pr8, src=src)
    return out


def _to_u8(img: torch.Tensor) -> np.ndarray:
    """float k/255 map -> uint8 (exact for values the bake wrote)"""
    return np.clip(np.rint(img.detach().float().cpu().numpy() * 255.0), 0, 255).astype(np.uint8)


def write_obj(directory: str, result: Dict[str, Any], texture_format: str = "jpg", name: str = "model") -> str:
    """Write `<name>.obj` (+ `<name>.mtl` and texture images) the way threestudio's saver does, for users running without
    threestudio.  `result` is what bake_textures returns (optionally with v_nrm / v_rgb) or the `params` of the exporter's
    ExporterOutput.  vt lines hold (u, 1 - v) and images are stored with row 0 (v = 0) at the top of the file, so
    OBJ's bottom-left texture origin addresses the texel the bake wrote.  Returns the .obj path."""
    import cv2
    if "mesh" in result:
        m = result["mesh"]
        texture_format = result.get("map_format") or texture_format
        result = {k: getattr(m, k) for k in ("v_pos", "t_pos_idx", "v_nrm", "v_tex", "t_tex_idx", "v_rgb")} | {
            k: result.get(k) for k in ("map_Kd", "map_Pm", "map_Pr")}
    os.makedirs(directory, exist_ok=True)
    obj = os.path.join(directory, f"{name}.obj")
    v = result["v_pos"].detach().cpu().numpy()
    f = result["t_pos_idx"].detach().cpu().numpy().astype(np.int64) + 1
    vn = result.get("v_nrm")
    vt, ft = result.get("v_tex"), result.get("t_tex_idx")
    rgb = result.get("v_rgb")
    maps = {k: result.get(k) for k in ("map_Kd", "map_Pm", "map_Pr")}
    lines = []
    if any(m is not None for m in maps.values()):
        lines += [f"mtllib {name}.mtl", "usemtl default"]
    if rgb is not None:
        rgb = rgb.detach().cpu().numpy()
        lines += [f"v {p[0]:.6f} {p[1]:.6f} {p[2]:.6f} {c[0]:.6f} {c[1]:.6f} {c[2]:.6f}" for p, c in zip(v, rgb)]
    else:
        lines += [f"v {p[0]:.6f} {p[1]:.6f} {p[2]:.6f}" for p in v]
    if vn is not None:
        lines += [f"vn {p[0]:.6f} {p[1]:.6f} {p[2]:.6f}" for p in vn.detach().cpu().numpy()]
    if vt is not None:
        vt = vt.detach().cpu().numpy().astype(np.float64)
        ft = ft.detach().cpu().numpy().astype(np.int64) + 1
        lines += [f"vt {p[0]:.8f} {1.0 - p[1]:.8f}" for p in vt]
    for i, t in enumerate(f):
        if vt is not None and vn is not None:
            lines.append("f " + " ".join(f"{t[k]}/{ft[i, k]}/{t[k]}" for k in range(3)))
        elif vt is not None:
            lines.append("f " + " ".join(f"{t[k]}/{ft[i, k]}" for k in range(3)))
        elif vn is not None:
            lines.append("f " + " ".join(f"{t[k]}//{t[k]}" for k in range(3)))
        else:
            lines.append(f"f {t[0]} {t[1]} {t[2]}")
    with open(obj, "w") as fh:
        fh.write("\n".join(lines) + "\n")
    if any(m is not None for m in maps.values()):
        mtl = ["newmtl default", "Ka 0.0 0.0 0.0", "Ks 0.0 0.0 0.0"]
        if maps["map_Kd"] is None:
            mtl.append("Kd 0.5 0.5 0.5")
        for key, fname in (("map_Kd", "texture_kd"), ("map_Pm", "texture_metallic"), ("map_Pr", "texture_roughness")):
            img = maps[key]
            if img is None:
                continue
            mtl.append(f"{key} {fname}.{texture_format}")
            u8 = _to_u8(img)
            u8 = cv2.cvtColor(u8, cv2.COLOR_RGB2BGR) if u8.shape[-1] == 3 else u8[..., 0]
            if not cv2.imwrite(os.path.join(directory, f"{fname}.{texture_format}"), u8):
                raise IOError(f"cv2 could not write {fname}.{texture_format}")
        with open(os.path.join(directory, f"{name}.mtl"), "w") as fh:
            fh.write("\n".join(mtl) + "\n")
    return obj
