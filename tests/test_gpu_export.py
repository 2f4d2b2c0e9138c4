"""GPU: the mesh exporter's texture bake (csrc/texbake.cu via dreammat_b200/texbake.py) against its CPU restatement
(oracle/export.py), and the `mesh-exporter` plugin end to end through the stub registry and write_obj."""
import os
import sys

import numpy as np
import pytest
import torch

from oracle import export as OE
from oracle import render as OR
from tests.test_plugin_registry import STUB, YAML_GEOMETRY, YAML_MATERIAL, _write_obj

pytestmark = pytest.mark.gpu

T = 256


def _seeded_geometry(geo, seed=0):
    """hash-grid and MLP parameters scaled so that the features are far from 0 (the default init gives ~1e-4).  Level l has
    amplitude 2^-l: with equal amplitudes the finest levels dominate and fp32 rounding of the grid coordinate alone moves
    ~1.5 % of the quantised texels by one step against the float64 oracle."""
    from dreammat_b200 import render_ops as R
    g = torch.Generator().manual_seed(seed)
    _, offs = R.hashgrid_num_params(geo.hg)
    amp = torch.cat([torch.full((2 * (offs[l + 1] - offs[l]),), 0.5 ** l) for l in range(len(offs) - 1)])
    geo.grid.copy_(((torch.rand(geo.n_grid, generator=g) * 2 - 1) * amp).to(geo.grid.device))
    geo.W1.mul_(4.0)
    geo.W2.mul_(4.0)


@pytest.fixture(scope="module")
def baked():
    from dreammat_b200 import system as Y
    from dreammat_b200 import texbake as TB
    v, f = OR.icosphere(3, bump=0.12)
    geo = Y.DreamMatMesh(device="cuda", mesh=(v, f))
    _seeded_geometry(geo)
    mat = Y.DreamMatMaterial(device="cuda")
    res = TB.bake_textures(geo, mat, T, 2, return_debug=True)
    torch.cuda.synchronize()
    a = res["atlas"]
    ref = OE.bake(a.uv_fixed, a.t_tex_idx, T, v.numpy(), f.numpy(), geo.grid.cpu(), geo.W1.cpu(), geo.W2.cpu())
    return geo, mat, res, ref


def test_raster_matches_oracle(baked):
    _, _, res, ref = baked
    owner = res["owner"].cpu().numpy()
    assert np.array_equal(owner, ref["owner"])
    cov = owner >= 0
    assert np.array_equal(res["mask"].cpu().numpy().astype(bool), cov)
    assert np.abs(res["bary"].cpu().numpy()[cov].astype(np.float64) - ref["bary"][cov]).max() <= 1e-7


def test_covered_texels_match_oracle(baked):
    _, _, res, ref = baked
    assert np.array_equal(res["texels"].cpu().numpy(), ref["texels"])
    assert np.abs(res["points"].cpu().numpy().astype(np.float64) - ref["points"]).max() <= 1e-6
    assert np.abs(ref["features"]).mean() > 0.2                   # the features are not ~0: the activations are exercised
    tex = ref["texels"]
    ours = np.concatenate([res["kd8"].cpu().numpy()[tex], res["pm8"].cpu().numpy()[tex, None], res["pr8"].cpu().numpy()[tex, None]], 1)
    d = np.abs(ours.astype(np.int64) - ref["maps"][tex])
    fe = np.abs(res["features"].cpu().numpy().astype(np.float64) - ref["features"]).max()
    assert d.max() <= 1 and (d.max(1) > 0).mean() < 1e-3, (d.max(), (d.max(1) > 0).mean(), d.max(0), fe)


def test_fill_is_exact_nearest_covered_texel(baked):
    from scipy.spatial import cKDTree
    _, _, res, ref = baked
    src = res["src"].cpu().numpy().astype(np.int64)
    assert (src >= 0).all()                                       # no texel left empty
    cov = ref["owner"] >= 0
    assert cov[src].all() and np.array_equal(src[cov], np.nonzero(cov)[0]), (cov[src].mean(), (src[cov] != np.nonzero(cov)[0]).sum())
    idx = np.arange(T * T)
    d2 = (idx // T - src // T) ** 2 + (idx % T - src % T) ** 2
    r2 = (idx // T - ref["src"] // T) ** 2 + (idx % T - ref["src"] % T) ** 2     # scipy's exact EDT
    assert np.array_equal(d2, r2), ((d2 != r2).sum(), (d2 - r2).min(), (d2 - r2).max())
    # values: k/255 of the source texel; where the nearest covered texel is unique it is the oracle's
    maps = torch.cat([res["map_Kd"], res["map_Pm"], res["map_Pr"]], -1).reshape(-1, 5).cpu().numpy()
    k = np.rint(maps * 255).astype(np.int64)
    assert np.array_equal(maps, (k / np.float32(255)).astype(np.float32))
    empty = np.nonzero(~cov)[0]
    pts = np.stack([np.nonzero(cov)[0] // T, np.nonzero(cov)[0] % T], 1)
    dd, _ = cKDTree(pts).query(np.stack([empty // T, empty % T], 1), k=2)
    uniq = empty[dd[:, 0] < dd[:, 1]]
    assert len(uniq) > 0.5 * len(empty), (len(uniq), len(empty))
    assert np.array_equal(src[uniq], ref["src"][uniq]), (src[uniq] != ref["src"][uniq]).sum()
    diff = np.abs(k[uniq] - ref["filled"][uniq].astype(np.int64))
    assert diff.max() <= 1 and (diff.max(1) > 0).mean() < 1e-2, (diff.max(), (diff.max(1) > 0).mean())


def test_bake_is_bit_reproducible(baked, tmp_path):
    from dreammat_b200 import texbake as TB
    geo, mat, res, _ = baked
    again = TB.bake_textures(geo, mat, T, 2, atlas=res["atlas"], return_debug=True)
    for key in ("owner", "bary", "mask", "texels", "points", "features", "src", "map_Kd", "map_Pm", "map_Pr"):
        assert torch.equal(res[key], again[key]), key
    tex = res["texels"].long()
    for key in ("kd8", "pm8", "pr8"):           # the uint8 maps are defined on the covered texels only
        assert torch.equal(res[key][tex], again[key][tex]), key
    files = []
    for i, r in enumerate((res, TB.bake_textures(geo, mat, T, 2))):
        d = tmp_path / str(i)
        TB.write_obj(str(d), r, "png")
        files.append({n: (d / n).read_bytes() for n in sorted(os.listdir(d))})
    assert files[0] == files[1] and len(files[0]) == 5


def _registry():
    for m in [k for k in sys.modules if k == "threestudio" or k.startswith("threestudio.") or k == "dreammat_b200.threestudio_plugin"]:
        del sys.modules[m]
    sys.path.insert(0, STUB)
    import threestudio
    import dreammat_b200.threestudio_plugin  # noqa: F401
    return threestudio


def _unregister():
    sys.path.remove(STUB)
    for m in [k for k in sys.modules if k == "threestudio" or k.startswith("threestudio.") or k == "dreammat_b200.threestudio_plugin"]:
        del sys.modules[m]


def test_mesh_exporter_through_the_registry(tmp_path):
    from dreammat_b200.scene import synthetic_envmap
    from dreammat_b200.texbake import write_obj
    threestudio = _registry()
    try:
        obj = tmp_path / "in.obj"
        _write_obj(str(obj))
        geo = threestudio.find("dreammat-mesh")(dict(YAML_GEOMETRY, shape_init=f"mesh:{obj}"))
        _seeded_geometry(geo.impl, 1)
        mat = threestudio.find("dreammat-material")(YAML_MATERIAL, env_maps=[synthetic_envmap(16, 32, seed=i) for i in range(5)])
        E = threestudio.find("mesh-exporter")
        outs = E({"texture_size": T, "texture_format": "png", "context_type": "cuda"}, geometry=geo, material=mat, background=None)()
        assert len(outs) == 1 and outs[0].save_name == "model.obj" and outs[0].save_type == "obj"
        p = outs[0].params
        assert p["save_mat"] and p["save_uv"] and p["map_Kd"].shape == (T, T, 3) and p["map_Pr"].shape == (T, T, 1)
        path = write_obj(str(tmp_path / "out"), p)
        # read back what was written, in OBJ's own convention: vt (s, t) with t = 0 at the bottom row of the image
        import cv2
        vs, vts, fs = [], [], []
        for line in open(path):
            q = line.split()
            if q and q[0] == "v":
                vs.append([float(x) for x in q[1:4]])
            elif q and q[0] == "vt":
                vts.append([float(x) for x in q[1:3]])
            elif q and q[0] == "f":
                fs.append([[int(i) - 1 for i in c.split("/")] for c in q[1:]])
        vs, vts, fs = np.array(vs), np.array(vts), np.array(fs)
        d = tmp_path / "out"
        kd = cv2.cvtColor(cv2.imread(str(d / "texture_kd.png"), cv2.IMREAD_UNCHANGED), cv2.COLOR_BGR2RGB)
        pm = cv2.imread(str(d / "texture_metallic.png"), cv2.IMREAD_UNCHANGED)
        pr = cv2.imread(str(d / "texture_roughness.png"), cv2.IMREAD_UNCHANGED)
        H, W = pm.shape
        # the texel at each face's UV centroid; keep faces whose UV triangle contains that texel's centre with margin
        tuv = vts[fs[..., 1]]                                            # [F,3,2]
        cen = tuv.mean(1)
        col, row = np.floor(cen[:, 0] * W).astype(int), np.floor((1 - cen[:, 1]) * H).astype(int)
        ctr = np.stack([(col + 0.5) / W, 1 - (row + 0.5) / H], 1)
        e1, e2, e0 = tuv[:, 1] - tuv[:, 0], tuv[:, 2] - tuv[:, 0], ctr - tuv[:, 0]
        den = e1[:, 0] * e2[:, 1] - e1[:, 1] * e2[:, 0]
        w1 = (e0[:, 0] * e2[:, 1] - e0[:, 1] * e2[:, 0]) / den
        w2 = (e1[:, 0] * e0[:, 1] - e1[:, 1] * e0[:, 0]) / den
        w = np.stack([1 - w1 - w2, w1, w2], 1)
        own = (np.abs(den) > 0) & (w > 1e-3).all(1)
        assert own.mean() > 0.5
        p3 = np.einsum("fk,fkc->fc", w[own], vs[fs[own, :, 0]])
        m = mat.export(**geo.export(torch.from_numpy(p3).float().cuda()))
        want = np.floor(torch.cat([m["albedo"], m["metallic"], m["roughness"]], -1).double().cpu().numpy() * 255)
        got = np.concatenate([kd[row[own], col[own]], pm[row[own], col[own], None], pr[row[own], col[own], None]], 1)
        assert np.abs(got - want).max() <= 1
        # fmt obj: per-vertex albedo from the same export kernel
        o = E({"fmt": "obj"}, geometry=geo, material=mat, background=None)()[0].params
        assert o["save_vertex_color"] and not o["save_mat"]
        ref = mat.export(**geo.export(geo.impl.v_pos.cuda()))["albedo"].cpu()
        assert (o["mesh"].v_rgb - ref).abs().max() <= 1e-6
    finally:
        _unregister()
