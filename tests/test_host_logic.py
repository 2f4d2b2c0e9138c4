"""CPU tests of the host-side mirrors (a1 batch, schedules, prompt selection, plugin Config surface)."""
import json
import os

import pytest
import torch

from oracle import render as OR
from oracle import sd as OS

SURFACE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "plugin_config_surface.json")


def test_camera_batch_matches_oracle():
    from dreammat_b200.scene import DataConfig, FixCameraSet
    cams = FixCameraSet(DataConfig(width=48, height=48), torch.Generator().manual_seed(0))
    ids = torch.tensor([0, 17, 63, 127])
    c = cams.cameras(ids)
    o = OR.camera_batch(cams.elevation_deg[ids], cams.azimuth_deg[ids], cams.camera_distances[ids], cams.fovy_deg[ids], 48, 48)
    for k in ("rays_o", "rays_d", "mvp_mtx", "w2c", "c2w", "camera_positions"):
        assert torch.allclose(c[k], o[k], atol=1e-6), k
    # configs/dreammat.yaml:11-17 ranges
    assert float(cams.elevation_deg.min()) >= -20 and float(cams.elevation_deg.max()) <= 45
    assert float(cams.camera_distances.min()) >= 3 and float(cams.camera_distances.max()) <= 4
    assert float(cams.fovy_deg.min()) >= 25 and float(cams.fovy_deg.max()) <= 45
    # stratified azimuths: one per 360/128 degree bin (uncond.py:606-614)
    bins = torch.floor((cams.azimuth_deg + 180) / (360 / 128)).long()
    assert torch.equal(bins, torch.arange(128))
    v, e = cams.collate(torch.Generator().manual_seed(3), 8)
    assert v.shape == (8,) and int(v.max()) < 128 and int(e.max()) < 5


def test_schedules_match_reference_semantics():
    from dreammat_b200.guidance import C
    for val, step in (([0, -1.0, -0.5, 2000], 0), ([0, -1.0, -0.5, 2000], 1000), ([0, -1.0, -0.5, 2000], 5000),
                      ([500, 0.2, 0.02, 501], 500), ([500, 0.2, 0.02, 501], 501), (1.05, 10), ([0, 0.0, -0.5, 2000], 300)):
        assert C(val, 0, step) == OS.C(val, 0, step)
    assert C([0, -1.0, -0.5, 2000], 0, 1000) == -0.75


def test_prompt_direction_selection():
    """models/prompt_processors/base.py:281-312: side default, front |az|<45, back |az|>135, overhead el>60 (last wins)."""
    from dreammat_b200.guidance import PromptProcessorOutput
    z = torch.zeros(1, 77, 8)
    pu = PromptProcessorOutput(z, z, z, torch.zeros(4, 77, 8), torch.zeros(4, 77, 8))
    el = torch.tensor([0.0, 0.0, 0.0, 0.0, 70.0, 0.0])
    az = torch.tensor([90.0, 10.0, -44.0, 170.0, 10.0, -136.0])
    assert pu.direction_index(el, az, torch.ones(6)).tolist() == [0, 1, 1, 2, 3, 2]
    vd = torch.arange(4).float().view(4, 1, 1).expand(4, 77, 8)
    pu = PromptProcessorOutput(z, z, z + 9, vd, vd + 10)
    e = pu.get_text_embeddings(el[:2], az[:2], torch.ones(2), True, return_null_text_embeddings=True)
    assert e.shape == (6, 77, 8) and e[:, 0, 0].tolist() == [0, 1, 10, 11, 9, 9]      # [text | uncond | null]


def test_plugin_config_surface_matches_reference():
    """Same Config field names (and scalar defaults) as the reference plugins, so dreammat.yaml parses unchanged.
    The reference's Config blocks are recorded in tests/golden/plugin_config_surface.json."""
    from dreammat_b200.guidance import StableDiffusionLightGuidance
    from dreammat_b200.system import DreamMatMaterial
    with open(SURFACE) as f:
        surface = json.load(f)
    for cls, mine in (("StableDiffusionLightGuidance", StableDiffusionLightGuidance.Config), ("DreamMatMaterial", DreamMatMaterial.Config)):
        ref = surface[cls]
        assert len(ref["fields"]) >= 10
        inst = mine()
        for name in ref["fields"]:
            assert hasattr(inst, name), f"{cls}.Config lacks field {name}"
        for name, default in ref["defaults"].items():
            assert getattr(inst, name) == default, (cls, name, default, getattr(inst, name))


def test_procedural_mesh_and_normalisation():
    from dreammat_b200.scene import normalize_mesh, procedural_mesh, vertex_normals
    import numpy as np
    v, f = procedural_mesh(5000, 0.8, 0)
    assert 4000 < f.shape[0] < 30000 and abs(float(v.abs().max()) - 0.8) < 1e-6
    vn = vertex_normals(v, f)
    assert torch.allclose(vn.norm(dim=-1), torch.ones(v.shape[0]), atol=1e-5)
    assert float((vn * torch.nn.functional.normalize(v, dim=-1)).sum(-1).mean()) > 0.8      # outward facing
    # dreammat_mesh.py:163-197: centred, scaled to max |coord| = scale, +y up / +z front -> z up / x front
    pts = np.array([[0.0, 2.0, 0.0], [0.0, 0.0, 1.0], [0.0, -2.0, -1.0]])
    out = normalize_mesh(pts, 0.5, "+y", "+z")
    assert abs(np.abs(out).max() - 0.5) < 1e-12 and out[0, 2] > 0 and abs(out[0, 0]) < 1e-12


def test_geometry_checkpoint_keys_and_layout():
    """N2: `geometry.encoding.encoding.encoding.params` is tcnn's flat fp32 [12 599 920]; MLP weights [64,32] / [5,64]."""
    from dreammat_b200.scene import procedural_mesh
    from dreammat_b200.system import DreamMatMesh
    geo = DreamMatMesh({"shape_init": "p"}, "cpu", mesh=procedural_mesh(200, 0.8, 0))
    sd = geo.state_dict("geometry.")
    assert sd["geometry.encoding.encoding.encoding.params"].shape == (12599920,)
    assert sd["geometry.feature_network.layers.0.weight"].shape == (64, 32)
    assert sd["geometry.feature_network.layers.2.weight"].shape == (5, 64)
    ck = {k: torch.full_like(v, 0.5) for k, v in sd.items()}
    ck["geometry.albedo_predictor.0.weight_v"] = torch.zeros(3)      # dead reference parameter: ignored
    geo.load_state_dict(ck)
    assert float(geo.params.min()) == 0.5 == float(geo.params.max())  # the views alias the one flat buffer
    with pytest.raises(ValueError):
        geo.load_state_dict({k: v[:-1] if v.dim() == 1 else v for k, v in ck.items()})


def test_material_export_matches_reference_formula():
    """N2: dreammat_material.py:765-797 — bake-time maps use the squared-roughness range and sqrt(r2 + 1e-7)."""
    from dreammat_b200.system import DreamMatMaterial
    mat = DreamMatMaterial({}, "cpu")
    f = torch.randn(7, 5, generator=torch.Generator().manual_seed(0))
    out = mat.export(f)
    m = torch.sigmoid(f)
    assert set(out) == {"albedo", "metallic", "roughness"}
    assert torch.equal(out["albedo"], m[:, :3])
    assert torch.allclose(out["metallic"], m[:, 3:4] * 0.9)
    assert torch.allclose(out["roughness"], torch.sqrt(m[:, 4:5] * 0.89 + 0.01 + 1e-7))
    f8 = torch.randn(7, 8, generator=torch.Generator().manual_seed(1))
    b = mat.export(f8)["bump"]
    assert b.shape == (7, 3) and float(b.min()) >= 0 and float(b.max()) <= 1


def test_gemm_tile_plan_matches_measured_choices():
    """dm_gemm_plan is a pure query of choose_tile(): the kernel / tile width / split-K per layer shape that the sweeps in
    profiles/r01_tile_sweep.txt and r01_exp_splitk.txt selected (8-view batch = 24 UNet samples, one-view batch = 3)."""
    import ctypes as C
    import __graft_entry__ as g
    g.build()                                   # no-op when the library is up to date
    from dreammat_b200._cabi import lib
    L = lib()

    def plan(M, N, K, act=0):
        k, b, s = C.c_int(), C.c_int(), C.c_int()
        assert L.dm_gemm_plan(M, N, K, act, 0, C.byref(k), C.byref(b), C.byref(s)) == 0
        return ("pair" if k.value else "single", b.value, s.value)

    L.dm_gemm_set_workspace(C.c_void_p(16), L.dm_gemm_workspace_bytes())      # the query never dereferences it
    try:
        assert plan(98304, 320, 2880) == ("pair", 160, 1)          # UNet level 0 conv, N = 320: two exact 160-wide pair tiles
        assert plan(24576, 640, 5760) == ("pair", 256, 1)          # level 1: 256-wide pairs despite the padded third tile
        assert plan(6144, 1280, 11520) == ("pair", 256, 1)         # level 2
        assert plan(1536, 1280, 23040) == ("pair", 256, 2)         # 8x8 latents, 8 views: 30 pair tiles -> split-K 2
        assert plan(192, 1280, 11520) == ("pair", 256, 14)         # 8x8 latents, one view: 5 pair tiles -> split-K 14
        assert plan(768, 1280, 11520) == ("pair", 256, 4)          # 16x16 latents, one view
        assert plan(2097152, 128, 1152) == ("single", 128, 1)      # VAE 512^2 level, N = 128
        assert plan(98304, 2560, 320, act=3) == ("pair", 256, 1)   # FF projection with the fused GEGLU epilogue
        assert plan(192, 1280, 1280) == ("single", 64, 1)          # short K: the workspace pass would cost more than it saves
        assert plan(12288, 320, 2880) == ("single", 128, 1)        # level 0 at one view: too few tiles for 160-wide pairs
    finally:
        L.dm_gemm_set_workspace(None, 0)
    assert plan(192, 1280, 11520)[2] == 1                          # no caller-owned workspace -> no split-K


def test_weight_layouts_for_the_tensor_core_kernels():
    """Host-side weight preparation (pure torch, no GPU): the implicit-GEMM K order and the GEGLU row interleave must
    express the same linear maps as the diffusers layouts."""
    import torch.nn.functional as F
    from dreammat_b200 import dense_ops as D
    g = torch.Generator().manual_seed(0)
    # conv [Cout, Cin, 3, 3] -> [Cout, 9 * Cin_pad], K index = tap * Cin_pad + c with tap = kh * 3 + kw
    w = torch.randn(6, 5, 3, 3, generator=g)
    wg = D.conv_weight_to_gemm(w, cin_pad=8, cout_pad=0, dtype=torch.float32)
    assert wg.shape == (6, 72)
    x = torch.randn(2, 5, 7, 7, generator=g)
    xp = F.pad(x, (1, 1, 1, 1))
    cols = torch.zeros(2, 7, 7, 72)
    for kh in range(3):
        for kw in range(3):
            cols[..., (kh * 3 + kw) * 8:(kh * 3 + kw) * 8 + 5] = xp[:, :, kh:kh + 7, kw:kw + 7].permute(0, 2, 3, 1)
    assert torch.allclose(cols @ wg.t(), F.conv2d(x, w, padding=1).permute(0, 2, 3, 1), atol=1e-5)
    # GEGLU: diffusers computes hidden, gate = proj(x).chunk(2, -1); hidden * gelu(gate).  The fused epilogue reads the
    # projection in blocks of 64 columns = [32 value | 32 gate]
    Dh = 96
    wp, bp = torch.randn(2 * Dh, 16, generator=g), torch.randn(2 * Dh, generator=g)
    a = torch.randn(10, 16, generator=g)
    pr = a @ wp.t() + bp
    want = pr[:, :Dh] * F.gelu(pr[:, Dh:])
    pi = a @ D.geglu_interleave(wp).t() + D.geglu_interleave(bp)
    blk = pi.view(10, Dh // 32, 2, 32)
    got = (blk[:, :, 0] * F.gelu(blk[:, :, 1])).reshape(10, Dh)
    assert torch.allclose(got, want, atol=1e-6)
