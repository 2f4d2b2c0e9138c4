"""Pins the CPU oracle (and the host-side mirrors) against golden vectors produced by EXECUTING the reference's own
function bodies (tests/golden/make_golden.py lifts them out of /root/reference by AST and runs them on seeded inputs).
Runs anywhere: only tests/golden/reference_vectors.pt is read.

Tolerances: the oracle restates the same fp32 torch arithmetic, so agreement is at rounding level (1e-6 absolute /
relative); sums over many samples get 1e-5."""
import os

import pytest
import torch
import torch.nn.functional as F

from oracle import render as OR
from oracle import sd as OS

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_vectors.pt")


@pytest.fixture(scope="module")
def G():
    return torch.load(GOLD, weights_only=False)


def close(a, b, tol=1e-6):
    a, b = a.detach().double(), b.detach().double()
    return float((a - b).abs().max()) <= tol * (1.0 + float(b.abs().max()))


def test_collate_cameras_rays_and_draws(G):
    """a1: data/uncond.py:723-821 + utils/ops.py:179-292 executed by the generator."""
    gi, go = G["collate"]["in"], G["collate"]["out"]
    torch.manual_seed(gi["seed"])
    B = gi["B"]
    view_id = torch.floor(torch.rand(B) * gi["elevation_degs"].shape[0]).long()     # :724
    env_id = torch.floor(torch.rand(B) * gi["lightmaps"].shape[1]).long()           # :797 (the next draw)
    assert torch.equal(view_id, go["view_id"]) and torch.equal(env_id, go["env_id"])
    c = OR.camera_batch(gi["elevation_degs"][view_id], gi["azimuth_degs"][view_id], gi["fix_camera_distances"][view_id],
                        gi["fovy_degs"][view_id], gi["H"], gi["W"])
    for k in ("rays_o", "rays_d", "mvp_mtx", "c2w", "w2c", "camera_positions"):
        assert close(c[k], go[k]), k
    assert close(gi["elevation_degs"][view_id], go["elevation"]) and close(gi["azimuth_degs"][view_id], go["azimuth"])
    # channel order of the condition map: [depth | normal | 6 x RGB light] (:799-802)
    cm = torch.cat((gi["depths"][view_id], gi["normals"][view_id], gi["lightmaps"][view_id, env_id]), -1)
    assert torch.equal(cm, go["condition_map"]) and cm.shape[-1] == 22
    # the product's host mirror draws the same ids from the same stream
    from dreammat_b200.scene import DataConfig, FixCameraSet
    cams = FixCameraSet(DataConfig(width=gi["W"], height=gi["H"], fix_view_num=gi["elevation_degs"].shape[0], fix_env_num=gi["lightmaps"].shape[1]),
                        torch.Generator().manual_seed(0))
    v2, e2 = cams.collate(torch.Generator().manual_seed(gi["seed"]), B)
    assert torch.equal(v2, go["view_id"]) and torch.equal(e2, go["env_id"])
    # ... and builds the same cameras / rays / matrices for them (scene.FixCameraSet.cameras = uncond.py:740-796)
    cams.elevation_deg, cams.azimuth_deg = gi["elevation_degs"], gi["azimuth_degs"]
    cams.camera_distances, cams.fovy_deg = gi["fix_camera_distances"], gi["fovy_degs"]
    pc = cams.cameras(v2)
    for k in ("rays_o", "rays_d", "mvp_mtx", "c2w", "w2c", "camera_positions", "elevation", "azimuth", "camera_distances"):
        assert close(pc[k], go[k]), k


def test_fixed_view_set_draw_order(G):
    """a1: set_fix_elevs / azims / camera_distance / *_perturb / fovy in the order of __init__ (uncond.py:584-645,692-698):
    with the reference's seed the product's FixCameraSet is the reference's camera set, fovy included (it is drawn after the
    three zero-scaled perturb draws)."""
    from dreammat_b200.scene import DataConfig, FixCameraSet
    g = G["fixed_views"]
    cams = FixCameraSet(DataConfig(width=32, height=32), torch.Generator().manual_seed(g["seed"]))
    assert close(cams.elevation_deg, g["elevation_degs"]) and close(cams.azimuth_deg, g["azimuth_degs"])
    assert close(cams.camera_distances, g["camera_distances"]) and close(cams.fovy_deg, g["fovy_degs"])


def test_condition_map_files_decode_like_the_reference(G, tmp_path):
    """a1 / N1: the reference's nested loadrgb / loaddepth (data/uncond.py:532-557) executed on PNG files; FixViewMaps reads the
    same files (reference directory layout), keeps RGB as uint8 and must reproduce the float maps bit for bit."""
    cv2 = pytest.importorskip("cv2")
    import numpy as np
    from dreammat_b200.scene import FixViewMaps
    g = G["maps"]
    for sub in ("depth", "normal", "light"):
        (tmp_path / sub).mkdir()
    cv2.imwrite(str(tmp_path / "depth" / "000.png"), g["depth_png_u16"].numpy().astype(np.uint16))
    cv2.imwrite(str(tmp_path / "normal" / "000.png"), g["rgb_png_u8"]["normal"].numpy())
    for tag in FixViewMaps.LIGHT_TAGS:
        cv2.imwrite(str(tmp_path / "light" / f"000_{tag}_env1.png"), g["rgb_png_u8"][tag].numpy())
    maps = FixViewMaps(str(tmp_path), 1, 1, g["size"], g["size"])
    cm = maps.condition_map(torch.tensor([0]), torch.tensor([0]))
    assert cm.shape == (1, g["size"], g["size"], 22)
    assert torch.equal(cm[0, ..., 0:1], g["depth"])
    assert torch.equal(cm[0, ..., 1:4], g["rgb"]["normal"])
    for i, tag in enumerate(FixViewMaps.LIGHT_TAGS):
        assert torch.equal(cm[0, ..., 4 + 3 * i: 7 + 3 * i], g["rgb"][tag]), tag
    assert maps.lightmaps.dtype == torch.uint8 and maps.normals.dtype == torch.uint8


def test_contract_to_unisphere_is_affine_for_radius_one(G):
    """a3: geometry/base.py:20-32 (bounded): the hash-grid input is (x - bmin) / (bmax - bmin); the oracle's
    geometry_forward and the CUDA kernel use exactly this map for radius 1."""
    g = G["contract"]
    assert close((g["x"] - g["bbox"][0]) / (g["bbox"][1] - g["bbox"][0]), g["out"])
    assert close((g["x"] + 1) / 2, g["out"])


def test_jitter_and_tangent_frame(G):
    """a3: raytracing_renderer.py:161-173 (the inline block, executed verbatim) and :306-316."""
    g = G["jitter"]
    sel = g["selector"]
    nrm, pos = g["gb_normal"][sel], g["gb_pos"][sel]
    assert close(OR.get_orthogonal_directions(nrm), g["ortho"])
    torch.manual_seed(g["seed"])
    n = pos.shape[0]
    ang = torch.rand(n, 1)                                                  # :164
    eps = torch.normal(mean=0.0, std=0.05, size=[n, 1])                     # :168
    assert close(OR.jitter_positions(pos, nrm, ang, eps), g["positions_jitter"])
    # the product draws N(0,1) * change_eps: same stream, same values
    torch.manual_seed(g["seed"])
    _ = torch.rand(n, 1)
    assert close(torch.randn(n, 1) * 0.05, eps)


def test_controlnet_normal_and_depth_maps(G):
    """a2: compute_controlnet_normals / compute_controlnet_depth (raytracing_renderer.py:326-343)."""
    g = G["controlnet_maps"]
    assert close(OR.controlnet_view_normals(g["normals"], g["w2c"][0]), g["normal_out"])
    assert close(OR.controlnet_depth(g["depth"], g["hit"]), g["depth_out"])


def _sphere_hit(occ):
    c = torch.tensor(occ["center"], dtype=torch.float32)
    r = occ["radius"]

    def fn(o, d):
        oc = o - c
        b = (oc * d).sum(-1)
        disc = b * b - ((oc * oc).sum(-1) - r * r)
        t = -b - torch.sqrt(disc.clamp_min(0))
        return (disc > 0) & (t > 0)
    return fn


def test_material_forward_backward_and_export(G):
    """a4: DreamMatMaterial.forward -> shade_raytracing (dreammat_material.py:713-763, 615-677, 490-604) executed with the
    reference's own sampling tables, an analytic occluder as ray tracer and a synthetic lat-long map; colour, the seven aux
    maps, mat_reg and the autograd gradients w.r.t. both feature tensors."""
    g = G["material"]
    gi, go = g["in"], g["out"]
    assert close(OR.direction_tables(gi["n_diffuse"]), gi["tab_d"]) and close(OR.direction_tables(gi["n_specular"]), gi["tab_s"])
    from dreammat_b200 import render_ops as R          # the tables the CUDA shader is fed (host side, numpy)
    assert close(R.direction_tables(gi["n_diffuse"]), gi["tab_d"]) and close(R.direction_tables(gi["n_specular"]), gi["tab_s"])
    f = gi["features"].clone().requires_grad_(True)
    fj = gi["features_jitter"].clone().requires_grad_(True)
    al, me, ro, reg = OR.material_params(f, fj)
    out = OR.shade_raytracing(gi["pts"], gi["normals"], gi["viewdirs"], gi["env"], me, ro, al, gi["rand_d"], gi["rand_s"],
                              _sphere_hit(gi["occluder"]), n_diffuse=gi["n_diffuse"], n_specular=gi["n_specular"])
    assert 0.05 < float(out["_hit"].float().mean()) < 0.95          # the occluder matters
    for k in ("color", "albedo", "roughness", "metalness", "specular_lights", "diffuse_lights", "specular_colors", "diffuse_colors"):
        assert close(out[k], go[k], 2e-6), k
    assert close(reg, go["mat_reg"])
    ((out["color"] * gi["cotangent"]).sum() + gi["reg_weight"] * reg).backward()
    assert close(f.grad, go["d_features"], 1e-5) and close(fj.grad, go["d_features_jitter"], 1e-5)
    # export (dreammat_material.py:765-797) through the product's host mirror
    from dreammat_b200.system import DreamMatMaterial
    ex = DreamMatMaterial({"use_bump": False}, "cpu").export(gi["features"])
    for k in ("albedo", "metallic", "roughness"):
        assert close(ex[k], g["export"][k]), k


def test_csd_combination_loss_and_gradient(G):
    """a8/a9: compute_grad_sds (dreammat_guidance.py:440-497) and the __call__ tail (:584-602) executed with fixed noise
    predictions: w(t), the CSD combination, nan_to_num, loss_sds = 0.5 * sum((z - sg(z - grad))^2) / B, d loss / d z = grad / B."""
    g = G["guidance"]
    gi, go = g["in"], g["out"]
    assert close(OS.alphas_cumprod(), gi["alphas"], 1e-6)
    c, u, n, s = gi["scales"]
    grad = OS.sds_grad(gi["eps_text"], gi["eps_uncond"], gi["eps_null"], gi["noise"], gi["t"], gi["alphas"], c, u, n, s)
    B = grad.shape[0]
    assert close(grad.norm(), go["grad_norm"])
    z = gi["latents"].clone().requires_grad_(True)
    loss = 0.5 * F.mse_loss(z, (z - grad).detach(), reduction="sum") / B
    assert close(loss, go["loss_sds"], 1e-5)
    loss.backward()
    assert close(z.grad, go["d_latents"]) and close(grad / B, go["d_latents"])
    norms = {"uncond_m_noise_norm": gi["eps_uncond"] - gi["noise"], "text_m_noise_norm": gi["eps_text"] - gi["noise"],
             "text_m_uncond_norm": gi["eps_text"] - gi["eps_uncond"], "text_m_null_norm": gi["eps_text"] - gi["eps_null"],
             "null_m_uncond_norm": gi["eps_null"] - gi["eps_uncond"], "noise_norm": gi["noise"], "uncond_norm": gi["eps_uncond"],
             "text_norm": gi["eps_text"]}
    for k, v in norms.items():
        assert close(v.norm(), go[k]), k


def test_prompt_selection_and_cfg_branch_layout(G):
    """a8: view-dependent embedding selection (prompt_processors/base.py:52-85 with the direction conditions of :243-309,
    executed) and the CFG batch layout of the UNet call (dreammat_guidance.py:388-438): [text | uncond | null]."""
    from dreammat_b200.guidance import PromptProcessorOutput, alphas_cumprod
    g = G["prompt"]
    t = g["tables"]
    pu = PromptProcessorOutput(t["text"], t["uncond"], t["null"], t["text_vd"], t["uncond_vd"])
    el, az = g["elevation"], g["azimuth"]
    assert torch.equal(pu.get_text_embeddings(el, az, torch.ones_like(el), True, return_null_text_embeddings=True), g["vd"])
    assert torch.equal(pu.get_text_embeddings(el, az, torch.ones_like(el), False, return_null_text_embeddings=True), g["no_vd"])
    b = G["branches"]
    B = b["latents_noisy"].shape[0]
    assert torch.equal(b["unet_in"], torch.cat([b["latents_noisy"]] * 3)) and torch.equal(b["unet_t"], torch.cat([b["t"]] * 3))
    assert torch.equal(b["unet_ctx"], pu.get_text_embeddings(el[:B], az[:B], torch.ones(B), True, return_null_text_embeddings=True))
    out = b["unet_in"] * 2 + b["unet_ctx"].mean(dim=(1, 2)).view(-1, 1, 1, 1)          # the generator's stand-in UNet
    for k, chunk in zip(("eps_text", "eps_uncond", "eps_null"), out.chunk(3)):
        assert torch.equal(chunk, b[k]), k
    assert close(alphas_cumprod(), G["guidance"]["in"]["alphas"])


def test_feature_mlp_structure_and_forward(G):
    """a3: VanillaMLP (models/networks.py:150-187) instantiated with dreammat.yaml's mlp_network_config: bias-free
    Linear -> ReLU -> Linear; its state-dict keys are the checkpoint keys DreamMatMesh.state_dict uses."""
    g = G["mlp"]
    sd = g["state_dict"]
    assert sorted(sd) == ["layers.0.weight", "layers.2.weight"]
    assert tuple(sd["layers.0.weight"].shape) == (64, 32) and tuple(sd["layers.2.weight"].shape) == (5, 64)
    assert close(OR.mlp_forward(g["enc"], sd["layers.0.weight"], sd["layers.2.weight"]), g["out"])


def test_schedule_C(G):
    """utils/misc.py:65-86 against the oracle's and the product's C()."""
    from dreammat_b200.guidance import C
    for (v, e, s, want) in G["C"]:
        assert abs(OS.C(v, e, s) - want) < 1e-12 and abs(C(v, e, s) - want) < 1e-12, (v, e, s)


def test_mesh_normalisation_block(G):
    """dreammat_mesh.py:163-197 executed verbatim (centre, up/front alignment, scale to shape_init_params) vs scene.normalize_mesh."""
    from dreammat_b200.scene import normalize_mesh
    g = G["mesh_normalize"]
    for (up, front, sc, want) in g["cases"]:
        got = normalize_mesh(g["vertices"].numpy().copy(), sc, up, front)
        assert float(abs(torch.from_numpy(got) - want).max()) < 1e-12, (up, front)


def test_vertex_normals(G):
    """models/mesh.py:135-161 against the oracle and the product's scene.vertex_normals."""
    from dreammat_b200.scene import vertex_normals
    g = G["vertex_normals"]
    assert close(OR.vertex_normals(g["v"], g["f"]), g["out"]) and close(vertex_normals(g["v"], g["f"]), g["out"])
