"""Mesh exporter, host side, no GPU: the UV atlas (dreammat_b200/uvatlas.py), the integer fill rule shared by the
rasterisers, the OBJ writer and the `mesh-exporter` plugin's configuration surface."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import export as OE
from oracle import render as OR
from dreammat_b200 import uvatlas as U
from tests.test_plugin_registry import YAML_GEOMETRY, _write_obj, stub_on_path  # noqa: F401

T, PAD = 256, 2


def _two_parts_and_a_zero_area_face():
    v1, f1 = OR.icosphere(1, 0.35)
    v2, f2 = OR.icosphere(1, 0.3, bump=0.1)
    v = np.concatenate([v1.numpy() - [0.45, 0, 0], v2.numpy() + [0.45, 0.1, 0]])
    f = np.concatenate([f1.numpy(), f2.numpy() + len(v1)])
    extra = np.array([[0.0, 0.7, 0.0], [0.1, 0.7, 0.0], [0.2, 0.7, 0.0]])       # collinear: zero area
    f = np.concatenate([f, [[len(v), len(v) + 1, len(v) + 2]]])
    return np.concatenate([v, extra]).astype(np.float32), f.astype(np.int32)


def helicoid(n_u=6, n_t=96, turns=2.0, pitch=0.12):
    """a ruled surface winding twice around its axis: its +-z charts fold over themselves in projection"""
    u = np.linspace(0.15, 0.8, n_u)
    t = np.linspace(0.0, 2 * np.pi * turns, n_t)
    U_, T_ = np.meshgrid(u, t, indexing="ij")
    v = np.stack([U_ * np.cos(T_), U_ * np.sin(T_), pitch * T_ - pitch * np.pi * turns], -1).reshape(-1, 3)
    idx = np.arange(n_u * n_t).reshape(n_u, n_t)
    a, b, c, d = idx[:-1, :-1], idx[1:, :-1], idx[1:, 1:], idx[:-1, 1:]
    f = np.concatenate([np.stack([a, b, c], -1).reshape(-1, 3), np.stack([a, c, d], -1).reshape(-1, 3)])
    return v.astype(np.float32), f.astype(np.int32)


MESHES = {"icosphere": lambda: tuple(x.numpy() for x in OR.icosphere(3, bump=0.12)),
          "two_parts_zero_area": _two_parts_and_a_zero_area_face, "helicoid": helicoid}


@pytest.mark.parametrize("name", sorted(MESHES))
def test_atlas_is_overlap_free_padded_uniform_and_deterministic(name):
    v, f = MESHES[name]()
    a = U.build_atlas(v, f, T, PAD)
    assert a.v_tex.dtype == np.float32 and a.t_tex_idx.shape == f.shape and a.uv_fixed.dtype == np.int32
    assert np.array_equal(a.v_tex, a.uv_fixed / (256.0 * T))
    assert a.v_tex.min() >= PAD / T and a.v_tex.max() <= 1 - PAD / T
    # faces of one chart share their corners; no vt is shared between charts
    owner_chart = np.full(len(a.v_tex), -1)
    owner_chart[a.t_tex_idx.reshape(-1)] = np.repeat(a.face_chart, 3)
    assert (owner_chart[a.t_tex_idx] == a.face_chart[:, None]).all()
    # the integer raster covers no texel centre twice (the restated raster of oracle/export.py)
    owner, _, count = OE.raster(a.uv_fixed, a.t_tex_idx, T)
    assert count.max() == 1 and (owner >= 0).sum() > 0.02 * T * T
    # chart masks dilated by `padding` (square structuring element) are disjoint
    cov = np.nonzero(owner >= 0)[0]
    ch = a.face_chart[owner[cov]]
    r, c = cov // T, cov % T
    dil = []
    for dr in range(-PAD, PAD + 1):
        for dc in range(-PAD, PAD + 1):
            dil.append(np.stack([ch, (r + dr) * (T + 2 * PAD) + (c + dc)], 1))
    dil = np.unique(np.concatenate(dil), axis=0)
    assert len(np.unique(dil[:, 1])) == len(dil), "dilated chart masks overlap"
    # one texel density: UV area = s^2 * projected area for every chart, up to the snapping of the corners
    v64, f64 = v.astype(np.float64), f.astype(np.int64)
    n = np.cross(v64[f64[:, 1]] - v64[f64[:, 0]], v64[f64[:, 2]] - v64[f64[:, 0]])
    proj_area = np.abs(n).max(1) / 2
    P = a.uv_fixed[a.t_tex_idx].astype(np.float64) / 256.0
    uv_area = ((P[:, 1, 0] - P[:, 0, 0]) * (P[:, 2, 1] - P[:, 0, 1]) - (P[:, 2, 0] - P[:, 0, 0]) * (P[:, 1, 1] - P[:, 0, 1])) / 2
    perim = np.linalg.norm(P - np.roll(P, 1, 1), axis=-1).sum(1)
    s2 = a.density ** 2
    for k in np.unique(a.face_chart):
        sel = a.face_chart == k
        bound = (perim[sel] * (2 ** 0.5 / 512) + 1e-6).sum()
        assert abs(uv_area[sel].sum() - s2 * proj_area[sel].sum()) <= bound, (name, k)
    # deterministic
    b = U.build_atlas(v, f, T, PAD)
    for x, y in ((a.v_tex, b.v_tex), (a.t_tex_idx, b.t_tex_idx), (a.uv_fixed, b.uv_fixed), (a.face_chart, b.face_chart)):
        assert np.array_equal(x, y)
    if name == "helicoid":           # the folded charts were split into one chart per face
        assert len(np.unique(a.face_chart)) > len(np.unique(U.charts_of(f64, U.face_classes(v64, f64))))


@pytest.mark.parametrize("diag", ["main", "anti"])
def test_two_triangles_of_a_square_cover_each_centre_once(diag):
    """Square with corners on texel centres: edges and diagonal pass through centres.  The top-left rule gives every
    centre of the half-open square (c0, c1] x (r0, r1] exactly one owner, in both rasterisers."""
    c0, c1, r0, r1 = 3, 12, 5, 14
    corners = np.array([[c0, r0], [c1, r0], [c1, r1], [c0, r1]]) * 256 + 128
    tri = np.array([[0, 1, 2], [0, 2, 3]] if diag == "main" else [[0, 1, 3], [1, 2, 3]])
    want = np.zeros((32, 32), np.int64)
    want[r0 + 1:r1 + 1, c0 + 1:c1 + 1] = 1
    owner, _, count = OE.raster(corners, tri, 32)
    assert np.array_equal(count.reshape(32, 32), want)
    tid, fid = U.raster_fixed(corners, tri, 32)
    assert np.array_equal(np.bincount(tid, minlength=32 * 32).reshape(32, 32), want)
    assert np.array_equal(owner[tid], fid)
    assert set(fid.tolist()) == {0, 1}


def test_atlas_rejects_bad_sizes_and_empty_meshes():
    v, f = OR.icosphere(1)
    for bad in (8, 8193):
        with pytest.raises(ValueError):
            U.build_atlas(v.numpy(), f.numpy(), bad)
    with pytest.raises(ValueError):
        U.build_atlas(v.numpy(), np.zeros((0, 3), np.int32), 64)


def test_bake_entry_points_reject_bad_sizes_and_empty_meshes():
    """argument checks run before any device work: a stand-in non-null pointer is never dereferenced"""
    import __graft_entry__ as g
    g.build()
    from dreammat_b200 import _cabi
    lib, p = _cabi.lib(), ctypes.c_void_p(16)
    for T in (8, 15, 8193):
        with pytest.raises(_cabi.DmError, match="texture size"):
            _cabi.check(lib.dm_uv_raster(p, p, 10, T, p, p, p, None), "dm_uv_raster")
        with pytest.raises(_cabi.DmError, match="texture size"):
            _cabi.check(lib.dm_seam_fill(p, T, p, p, p, p, p, p, p, p, None), "dm_seam_fill")
    with pytest.raises(_cabi.DmError, match="empty mesh"):
        _cabi.check(lib.dm_uv_raster(p, p, 0, 64, p, p, p, None), "dm_uv_raster")
    with pytest.raises(_cabi.DmError, match="no covered texel"):
        _cabi.check(lib.dm_texel_positions(p, 0, p, p, p, p, p, None), "dm_texel_positions")


def test_write_obj_round_trip(tmp_path):
    import cv2
    from dreammat_b200.texbake import write_obj
    g = torch.Generator().manual_seed(0)
    v, f = OR.icosphere(1)
    a = U.build_atlas(v.numpy(), f.numpy(), 64, PAD)
    k = {key: torch.randint(0, 256, (64, 64, c), generator=g) for key, c in (("map_Kd", 3), ("map_Pm", 1), ("map_Pr", 1))}
    res = {"v_pos": v, "t_pos_idx": f, "v_tex": torch.from_numpy(a.v_tex), "t_tex_idx": torch.from_numpy(a.t_tex_idx),
           **{key: x.float() / 255 for key, x in k.items()}}
    path = write_obj(str(tmp_path), res, "png")
    vs, vts, faces, mtllib = [], [], [], None
    for line in open(path):
        p = line.split()
        if p[0] == "v":
            vs.append([float(x) for x in p[1:4]])
        elif p[0] == "vt":
            vts.append([float(x) for x in p[1:3]])
        elif p[0] == "f":
            faces.append([[int(i) for i in q.split("/")] for q in p[1:]])
        elif p[0] == "mtllib":
            mtllib = p[1]
    faces = np.array(faces)
    assert np.allclose(np.array(vs), v.numpy(), atol=1e-6)
    assert np.array_equal(faces[..., 0] - 1, f.numpy()) and np.array_equal(faces[..., 1] - 1, a.t_tex_idx)
    vt = np.array(vts)
    assert np.allclose(vt[:, 0], a.v_tex[:, 0], atol=1e-7) and np.allclose(1 - vt[:, 1], a.v_tex[:, 1], atol=1e-7)
    mtl = dict(line.split(None, 1) for line in open(tmp_path / mtllib) if line.strip())
    files = {key: mtl[key].strip() for key in ("map_Kd", "map_Pm", "map_Pr")}
    kd = cv2.imread(str(tmp_path / files["map_Kd"]), cv2.IMREAD_UNCHANGED)
    assert np.array_equal(cv2.cvtColor(kd, cv2.COLOR_BGR2RGB), k["map_Kd"].numpy().astype(np.uint8))   # row 0 = v 0, top of file
    for key in ("map_Pm", "map_Pr"):
        img = cv2.imread(str(tmp_path / files[key]), cv2.IMREAD_UNCHANGED)
        assert img.ndim == 2 and np.array_equal(img, k[key][..., 0].numpy().astype(np.uint8))


def test_mesh_exporter_config_and_loud_rejections(stub_on_path, tmp_path):
    import threestudio
    import dreammat_b200.threestudio_plugin  # noqa: F401
    from threestudio.models.exporters.base import Exporter
    E = threestudio.find("mesh-exporter")
    assert E.__module__ == "dreammat_b200.threestudio_plugin" and issubclass(E, Exporter)
    c = E.Config()
    assert (c.save_video, c.fmt, c.save_name, c.save_normal, c.save_uv, c.save_texture, c.texture_size, c.texture_format,
            c.xatlas_chart_options, c.xatlas_pack_options, c.context_type) == \
        (False, "obj-mtl", "model", False, True, True, 1024, "jpg", {}, {}, "gl")
    obj = tmp_path / "m.obj"
    _write_obj(str(obj))
    geo = threestudio.find("dreammat-mesh")(dict(YAML_GEOMETRY, shape_init=f"mesh:{obj}"))
    mods = dict(geometry=geo, material=object(), background=None)
    for bad in ({"not_a_field": 1}, {"xatlas_chart_options": {"max_iterations": 2}}, {"xatlas_pack_options": {"resolution": 512}},
                {"save_uv": False}, {"fmt": "fbx"}):
        with pytest.raises(Exception):
            E(bad, **mods)
    with pytest.raises(ValueError, match="save_uv must be True"):
        E({"save_uv": False}, **mods)
    with pytest.raises(TypeError, match="exports its own geometry and material"):
        E({"xatlas_pack_options": {"padding": 4}, "context_type": "cuda"}, **mods)              # foreign material
    with pytest.raises(TypeError, match="exports its own geometry and material"):
        E({}, geometry=object(), material=object(), background=None)
