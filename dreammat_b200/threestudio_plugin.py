"""Drop-in plugin layer: registers the five hot-path plugins and the mesh exporter under the reference's registry names.

    import threestudio                      # the reference package (threestudio_dreammat/threestudio)
    import dreammat_b200.threestudio_plugin # re-registers the names below; last writer wins (threestudio/__init__.py:4-13)

    dreammat-system                      systems/dreammat.py:18-86            -> DreamMat
    dreammat-mesh                        models/geometry/dreammat_mesh.py:89  -> DreamMatMesh
    dreammat-material                    models/materials/dreammat_material.py:346 -> DreamMatMaterial
    raytracing-renderer                  models/renderers/raytracing_renderer.py:86 -> RaytraceRender
    stable-diffusion-dreammat-guidance   models/guidance/dreammat_guidance.py:44 -> StableDiffusionLightGuidance
    mesh-exporter                        models/exporters/mesh_exporter.py    -> MeshExporter (texbake.py)

Every class keeps the reference's construction protocol -- `cls(cfg, *args, **kwargs)` -> `parse_structured(Config, cfg)`
-> `configure(*args, **kwargs)` (utils/base.py:70-118; the system: systems/base.py:35-50) -- its Config field names /
defaults, call signatures, output keys and state-dict keys, so `launch.py` with `configs/dreammat.yaml` drives it
unchanged: the data module, prompt processor, background, Lightning trainer and logging stay the reference's; the exporter's
output goes through the host's own `save_obj`.

The classes derive from threestudio's own bases (BaseModule / BaseObject / BaseLift3DSystem): `isinstance(x, Updateable)`
keeps working, so the system's per-step `do_update_step` walk reaches `guidance.update_step` exactly as before.
"""
from __future__ import annotations

import dataclasses
import os
from dataclasses import dataclass, field
from typing import Any, Dict, List, Optional

import numpy as np
import torch
import torch.nn as nn

import threestudio
from threestudio.models.exporters.base import Exporter, ExporterOutput
from threestudio.systems.base import BaseLift3DSystem
from threestudio.utils.base import BaseModule, BaseObject

from . import guidance as _G
from . import render_ops as R
from . import scene as _S
from . import system as _Y
from . import texbake as _T
from . import weights as _W


def _plain(cfg, drop=("weights",)) -> dict:
    """structured config (OmegaConf DictConfig / dataclass instance / dict) -> plain dict for the host mirrors"""
    try:
        from omegaconf import OmegaConf
        if OmegaConf.is_config(cfg):
            cfg = OmegaConf.to_container(cfg, resolve=True)
    except ImportError:
        pass
    if dataclasses.is_dataclass(cfg) and not isinstance(cfg, type):
        cfg = dataclasses.asdict(cfg)
    return {k: v for k, v in dict(cfg).items() if k not in drop}


# ================================================================================================ geometry


class _Slot(nn.Module):
    """empty container: gives the trainable tensors the reference's state-dict paths"""


class _WNLinear(nn.Module):
    """Key-compatible stand-in for nn.utils.weight_norm(nn.Linear) (dreammat_mesh.py:62-74): bias / weight_g / weight_v.
    The reference builds three such predictors and never calls them (dead parameters, SURVEY.md section 2.1); they exist
    here only so that checkpoints round-trip with strict=True in both directions."""

    def __init__(self, fin, fout):
        super().__init__()
        v = torch.empty(fout, fin)
        nn.init.kaiming_uniform_(v, a=5 ** 0.5)
        self.bias = nn.Parameter(torch.zeros(fout), requires_grad=False)
        self.weight_g = nn.Parameter(v.norm(dim=1, keepdim=True), requires_grad=False)
        self.weight_v = nn.Parameter(v, requires_grad=False)


def _dead_predictor(fin, fout, run=256):
    return nn.Sequential(_WNLinear(fin, run), nn.ReLU(), _WNLinear(run, run), nn.ReLU(), _WNLinear(run, run), nn.ReLU(),
                         _WNLinear(run, fout))


@threestudio.register("dreammat-mesh")
class DreamMatMesh(BaseModule):
    @dataclass
    class Config(BaseModule.Config):
        # models/geometry/dreammat_mesh.py:93-121 (+ BaseExplicitGeometry.radius, geometry/base.py:191-193)
        radius: float = 1.0
        n_input_dims: int = 3
        n_feature_dims: int = 5
        pos_encoding_config: dict = field(default_factory=lambda: dict(_Y.DreamMatMesh.Config().pos_encoding_config))
        mlp_network_config: dict = field(default_factory=lambda: dict(_Y.DreamMatMesh.Config().mlp_network_config))
        shape_init: str = ""
        shape_init_params: Optional[Any] = None
        shape_init_mesh_up: str = "+z"
        shape_init_mesh_front: str = "+x"

    cfg: Config

    def configure(self, mesh=None) -> None:
        impl = _Y.DreamMatMesh(_plain(self.cfg), device=self.device, mesh=mesh)
        object.__setattr__(self, "impl", impl)                      # plain attribute: not a submodule
        # trainable tensors = views of impl's ONE flat buffer, exposed under the reference's parameter names
        # (encoding.encoding.encoding.params is tcnn's flat hash grid, feature_network.layers.{0,2}.weight the bias-free MLP)
        self.encoding = _Slot(); self.encoding.encoding = _Slot(); self.encoding.encoding.encoding = _Slot()
        self.encoding.encoding.encoding.params = nn.Parameter(impl.grid)
        self.feature_network = _Slot()
        l0, l2 = _Slot(), _Slot()
        l0.weight, l2.weight = nn.Parameter(impl.W1), nn.Parameter(impl.W2)
        self.feature_network.layers = nn.Sequential(l0, nn.ReLU(), l2)
        impl.bind_parameters(self.encoding.encoding.encoding.params, l0.weight, l2.weight)
        r = float(self.cfg.radius)
        self.register_buffer("bbox3d", torch.tensor([[-r] * 3, [r] * 3], dtype=torch.float32))
        self.register_buffer("bbox2d", torch.tensor([[-r] * 2, [r] * 2], dtype=torch.float32))
        pos_dim = 3 + 3 * 2 * 10                                     # get_embedder(10, 3), dreammat_mesh.py:50-61
        self.metallic_predictor = _dead_predictor(pos_dim, 1)
        self.roughness_predictor = _dead_predictor(pos_dim, 1)
        self.albedo_predictor = _dead_predictor(pos_dim, 3)
        self.register_buffer("v_buffer", impl.v_pos.clone())
        self.register_buffer("vnrm_buffer", impl.v_nrm.clone())
        self.register_buffer("vtex_buffer", impl.v_tex.clone())
        self.register_buffer("t_buffer", impl.t_pos_idx.long())

    # ---- the reference's geometry API
    def isosurface(self):
        return self.impl.isosurface()

    def forward(self, points, output_normal: bool = False) -> Dict[str, torch.Tensor]:
        return self.impl.forward(points, output_normal)

    def export(self, points, **kwargs) -> Dict[str, Any]:
        return self.impl.export(points, **kwargs)


# ================================================================================================ material


@threestudio.register("dreammat-material")
class DreamMatMaterial(BaseModule):
    @dataclass
    class Config(BaseModule.Config):
        # models/materials/dreammat_material.py:348-366
        material_activation: str = "sigmoid"
        environment_texture: str = "load/lights/mud_road_puresky_1k.hdr"
        environment_scale: float = 1.0
        min_metallic: float = 0.0
        max_metallic: float = 0.9
        min_roughness_squre: float = 0.01
        max_roughness_squre: float = 0.9
        min_roughness: float = 0.1
        max_roughness: float = 0.95
        use_bump: bool = True
        diffuse_sample_num: int = 512
        specular_sample_num: int = 256
        geometry_type: str = "schlick"
        random_azimuth: bool = True
        use_raytracing: bool = True

    cfg: Config
    requires_normal: bool = True        # models/materials/base.py:19-20 flags read by renderers
    requires_tangent: bool = False

    def configure(self, env_maps: Optional[List[torch.Tensor]] = None, fg_lut: Optional[torch.Tensor] = None) -> None:
        """dreammat_material.py:368-424: five lat-long maps `<environment_texture>/map{1..5}/map{1..5}.exr`, the FG LUT
        `load/lights/bsdf_256_256.bin`, and (split-sum branch) the prefiltered cube maps -- built on the device."""
        c = self.cfg
        if env_maps is None:
            env_maps = _S.load_reference_envmaps(c.environment_texture)
        if fg_lut is None and not c.use_raytracing:
            fg_lut = _S.load_fg_lut(os.path.join(os.path.dirname(c.environment_texture.rstrip("/")) or "load/lights", "bsdf_256_256.bin"))
        impl = _Y.DreamMatMaterial(_plain(c), device=self.device, env_maps=env_maps, fg_lut=fg_lut)
        object.__setattr__(self, "impl", impl)
        # state-dict parity with the reference module (dreammat_material.py:400-416): two buffers and one dead predictor
        tab = R.direction_tables(8192).double()                       # sample_sphere(8192, 0) -> az_el_to_points (:104-108)
        az, el = tab[:, 0] * 2 * np.pi, (1 - tab[:, 1]) * np.pi / 2
        self.register_buffer("light_pts", torch.stack([torch.cos(az) * torch.cos(el), torch.sin(az) * torch.cos(el), torch.sin(el)], -1).float())
        self.register_buffer("FG_LUT", (fg_lut if fg_lut is not None else torch.zeros(1, 256, 256, 2)).float().reshape(1, 256, 256, 2).clone())
        self.inner_light = _dead_predictor(3 + 3 * 2 * 8 + 72, 3)     # get_embedder(8, 3) + 72 IDE features (:412-415)
        self.inner_light.add_module("7", nn.Identity())               # the (parameter-free) ExpActivation slot

    def set_raytracer(self, raytracer):
        self.impl.set_raytracer(raytracer)

    def forward(self, pts, features, features_jitter, viewdirs, normals, env_id, **kwargs):
        return self.impl.forward(pts, features, features_jitter, viewdirs, normals, env_id, **kwargs)

    def export(self, features, **kwargs) -> Dict[str, Any]:
        return self.impl.export(features, **kwargs)


# ================================================================================================ renderer


@threestudio.register("raytracing-renderer")
class RaytraceRender(BaseModule):
    @dataclass
    class Config(BaseModule.Config):
        radius: float = 1.0           # models/renderers/base.py:17-18
        context_type: str = "gl"      # raytracing_renderer.py:88-90 (no rasteriser context is needed here)

    cfg: Config

    def configure(self, geometry, material, background=None) -> None:
        """systems/base.py:290-295 passes the three modules as keyword arguments; they are kept un-registered
        (renderers/base.py:22-35) so the renderer's state dict stays the reference's (`bbox` only)."""
        object.__setattr__(self, "sub_modules", (geometry, material, background))
        r = float(self.cfg.radius)
        self.register_buffer("bbox", torch.tensor([[-r] * 3, [r] * 3], dtype=torch.float32))
        impl = _Y.RaytraceRender(_plain(self.cfg), geometry=geometry.impl, material=material.impl, background=background,
                                 device=self.device)
        object.__setattr__(self, "impl", impl)

    @property
    def geometry(self):
        return self.sub_modules[0]

    @property
    def material(self):
        return self.sub_modules[1]

    @property
    def background(self):
        return self.sub_modules[2]

    def forward(self, env_id, rays_o, rays_d, w2c, mvp_mtx, camera_positions=None, light_positions=None, height=None,
                width=None, render_rgb: bool = True, **kwargs) -> Dict[str, Any]:
        return self.impl.forward(env_id, rays_o, rays_d, w2c, mvp_mtx, camera_positions, light_positions, height, width,
                                 view_id=kwargs.get("view_id"))


# ================================================================================================ guidance


def _find_safetensors(root: Optional[str], name: str, sub: Optional[str]) -> str:
    """Local resolution of a diffusers model id: `<cache_dir>/<name>[/<sub>]` or `<name>[/<sub>]` must hold
    *.safetensors (there is no network on the box; nothing is downloaded)."""
    cands = []
    for base in ([os.path.join(root, name)] if root else []) + [name] + ([root] if root else []):
        cands.append(os.path.join(base, sub) if sub else base)
    for c in cands:
        if os.path.isdir(c) and any(f.endswith(".safetensors") for f in os.listdir(c)):
            return c
    raise FileNotFoundError(f"no .safetensors found for '{name}' (looked in {cands}); dreammat_b200 loads diffusers-format "
                            "weights from local directories only")


@threestudio.register("stable-diffusion-dreammat-guidance")
class StableDiffusionLightGuidance(BaseObject):
    Config = _G.StableDiffusionLightGuidance.Config       # dreammat_guidance.py:45-84, field for field
    cfg: Config

    # hook for hosts without checkpoints (benchmarks, tests): callable(cfg) -> (unet_cfg, vae_cfg, w_unet, w_controlnet, w_vae)
    weight_source = None

    def configure(self) -> None:
        c = self.cfg
        if type(self).weight_source is not None:
            ucfg, vcfg, wu, wc, wv = type(self).weight_source(c)
        else:
            d_unet = _find_safetensors(c.cache_dir, c.pretrained_model_name_or_path, "unet")
            d_vae = _find_safetensors(c.cache_dir, c.pretrained_model_name_or_path, "vae")
            d_cn = _find_safetensors(None, c.controlnet_path, None) if c.use_controlnet else None
            # architecture from the checkpoints' own config.json (SD-2.1-base / the 22-channel ControlNet by default)
            ucfg = _W.unet_config_from_json(os.path.join(d_unet, "config.json"), os.path.join(d_cn, "config.json") if d_cn else None)
            vcfg = _W.vae_config_from_json(os.path.join(d_vae, "config.json"))
            wu, wv = _W.load_safetensors(d_unet), _W.load_safetensors(d_vae)
            wc = _W.load_safetensors(d_cn) if d_cn else None
        impl = _G.StableDiffusionLightGuidance(_plain(c, drop=()), ucfg, vcfg, wu, wc, wv, device=self.device)
        self.impl = impl

    def update_step(self, epoch: int, global_step: int, on_load_weights: bool = False):
        self.impl.update_step(epoch, global_step, on_load_weights)

    def __call__(self, rgb, prompt_utils, elevation, azimuth, camera_distances, env_id=None, rgb_as_latents=False, **kwargs):
        return self.impl(rgb, prompt_utils, elevation, azimuth, camera_distances, env_id, rgb_as_latents, **kwargs)


# ================================================================================================ system


class _FusedStepLoss(torch.autograd.Function):
    """Carries the gradient the fused kernel sequence already computed into torch's autograd, so that Lightning's
    `loss.backward()` + optimizer (systems/utils.py:34-53) run unchanged after `training_step`."""

    @staticmethod
    def forward(ctx, loss_value, scale_holder, grid, W1, W2, ggrid, gW1, gW2):
        ctx.save_for_backward(ggrid, gW1, gW2)
        return loss_value.clone()

    @staticmethod
    def backward(ctx, g):
        ggrid, gW1, gW2 = ctx.saved_tensors
        return None, None, ggrid * g, gW1 * g, gW2 * g, None, None, None


@threestudio.register("dreammat-system")
class DreamMat(BaseLift3DSystem):
    @dataclass
    class Config(BaseLift3DSystem.Config):
        # systems/dreammat.py:21-30
        texture: bool = True
        latent_steps: int = 1000
        save_train_image: bool = True
        save_train_image_iter: int = 1
        init_step: int = 0
        init_width: int = 512
        init_height: int = 512
        test_background_white: Optional[bool] = False
        # B200 addition: run the iteration as the explicit fused kernel sequence (system.DreamMat.training_step_fused)
        # instead of the op-by-op autograd graph; both give the same gradients
        fused_step: bool = True

    cfg: Config

    def configure(self) -> None:
        super().configure()      # geometry / material / background / renderer through threestudio.find (systems/base.py:243-295)

    def forward(self, batch: Dict[str, Any]) -> Dict[str, Any]:
        return {**self.renderer(**batch, render_rgb=self.cfg.texture)}

    def on_fit_start(self) -> None:
        super().on_fit_start()
        # systems/dreammat.py:44-50: built here because they are only used in training
        self.prompt_processor = threestudio.find(self.cfg.prompt_processor_type)(self.cfg.prompt_processor)
        self.guidance = threestudio.find(self.cfg.guidance_type)(self.cfg.guidance)
        g = getattr(self.guidance, "impl", self.guidance)
        impl = _Y.DreamMat({"loss": _plain(self.cfg.loss, ()), "optimizer": _plain(self.cfg.optimizer, ())}, self.geometry.impl,
                           self.material.impl, self.renderer.impl, g, None, device=self.geometry.impl.device)
        object.__setattr__(self, "impl", impl)
        from .parallel import quiesce_host_gc
        quiesce_host_gc()

    def _log(self, name, value):
        try:
            self.log(name, value)
        except Exception:      # outside a Trainer loop (tests, scripts) LightningModule.log is unavailable
            pass

    def _save_train_images(self, out, batch) -> None:
        """systems/dreammat.py:88-178: every `save_train_image_iter` steps one grid -- a row of eight render outputs and a row of
        the condition map's eight channel groups (depth | normal | six light maps).  Needs the host's saver mixin."""
        saver = getattr(self, "save_image_grid", None)
        step = int(self.true_global_step)
        if not self.cfg.save_train_image or saver is None or step % int(self.cfg.save_train_image_iter) != 0:
            return
        cell = DreamMat._cell
        renders = [cell(out[k][0], k in ("comp_depth", "metalness", "roughness"))
                   for k in ("comp_rgb", "specular_light", "diffuse_light", "comp_normal", "comp_depth", "albedo", "metalness", "roughness")]
        cm = batch["condition_map"][0]
        conditions = [cell(cm[:, :, 0:1], True)] + [cell(cm[:, :, c:c + 3]) for c in range(1, 22, 3)]
        saver(f"train/it{step}.png", imgs=[renders, conditions], name="train_step", step=step)

    def training_step(self, batch, batch_idx):
        """systems/dreammat.py:57-86."""
        prompt_utils = self.prompt_processor()
        step = int(self.true_global_step)
        if not self.cfg.fused_step or not self.cfg.texture:
            out = self(batch)
            batch["cond_normal"], batch["cond_depth"] = out.get("comp_normal"), out.get("comp_depth")
            guidance_out = self.guidance(out["comp_rgb"], prompt_utils, **batch, rgb_as_latents=False)
            loss = 0.0
            for name, value in guidance_out.items():
                if name.startswith("_"):
                    continue
                self._log(f"train/{name}", value)
                if name.startswith("loss_"):
                    loss = loss + value * self.C(self.cfg.loss[name.replace("loss_", "lambda_")])
            for name, value in out.items():
                if name.startswith("loss_"):
                    self._log(f"train/{name}", value)
                    loss = loss + value * self.C(self.cfg.loss[name.replace("loss_", "lambda_")])
            for name, value in self.cfg.loss.items():
                self._log(f"train_params/{name}", self.C(value))
            self._save_train_images(out, batch)
            return {"loss": loss}
        impl, geo = self.impl, self.geometry.impl
        impl.prompt_utils = prompt_utils
        impl.global_step = step                       # schedules (C(...)) follow the trainer's step counter
        out = impl.training_step_fused(batch, apply_optimizer=False)
        for k, v in out.items():      # same keys as the reference logs: loss_sds, grad_norm, the 8 diagnostic norms, loss_mat_reg
            if k.startswith("loss_") or k.endswith("_norm"):
                self._log(f"train/{k}", v)
        for name, value in self.cfg.loss.items():
            self._log(f"train_params/{name}", self.C(value))
        if (self.cfg.save_train_image and hasattr(self, "save_image_grid") and "condition_map" in batch
                and step % int(self.cfg.save_train_image_iter) == 0):
            with torch.no_grad():         # the fused step keeps no aux maps: the monitoring grid renders them on its (rare) steps
                self._save_train_images(self(batch), batch)
        p = self.geometry
        loss = _FusedStepLoss.apply(out["loss"], None, p.encoding.encoding.encoding.params, p.feature_network.layers[0].weight,
                                    p.feature_network.layers[2].weight, geo.dgrid, geo.dW1, geo.dW2)
        return {"loss": loss, "comp_rgb": out["comp_rgb"]}

    @staticmethod
    def _cell(img, gray=False):
        if gray:
            return {"type": "grayscale", "img": img[..., 0], "kwargs": {"cmap": None, "data_range": (0, 1)}}
        return {"type": "rgb", "img": img, "kwargs": {"data_format": "HWC", "data_range": (0, 1)}}

    def _grid(self, out, keys):
        cells = [self._cell(out["comp_rgb"][0].detach())] if self.cfg.texture else []
        return cells + [self._cell(out[k][0], k in ("metalness", "roughness")) for k in keys]

    def validation_step(self, batch, batch_idx=None):
        """systems/dreammat.py:181-240: one grid per validation view (render | lights | colours | normal | albedo | metalness | roughness)."""
        out = self(batch)
        step = self.true_global_step
        self.save_image_grid(f"validate/it{step}-{batch['index'][0]}.png",
                             self._grid(out, ("specular_light", "diffuse_light", "specular_color", "diffuse_color", "comp_normal", "albedo",
                                              "metalness", "roughness")), name="validation_step", step=step)

    def on_validation_epoch_end(self):
        pass

    def test_step(self, batch, batch_idx=None):
        """systems/dreammat.py:245-296: the per-view grid plus the four RGBA maps (albedo / roughness / metallic / render, alpha =
        opacity) the texture baker reads."""
        out = self(batch)
        step, idx = self.true_global_step, batch["index"][0]
        self.save_image_grid(f"it{step}-test/view/{idx}.png", self._grid(out, ("comp_normal", "albedo", "metalness", "roughness")),
                             name="test_step", step=step)
        mask = out["opacity"][0].detach()
        maps = {"albedo": out["albedo"][0].detach(), "roughness": out["roughness"][0].detach().repeat(1, 1, 3),
                "metallic": out["metalness"][0].detach().repeat(1, 1, 3), "render": out["comp_rgb"][0].detach()}
        for name, img in maps.items():
            self.save_img(torch.cat((img, mask), 2), f"it{step}-test/{name}/{idx}.png")

    def on_test_epoch_end(self):
        """systems/dreammat.py:298-300"""
        self.save_gif("it" + str(self.true_global_step) + "-test/view", fps=30)


# ================================================================================================ exporter


@threestudio.register("mesh-exporter")
class MeshExporter(Exporter):
    """threestudio's `mesh-exporter` (what `launch.py --export` builds from the system's default `exporter_type`) for this
    package's geometry and material: the atlas of uvatlas.py and the texture bake of texbake.py instead of xatlas,
    nvdiffrast and cv2.inpaint.  Returns one ExporterOutput that the host's `save_obj` writes unchanged."""

    @dataclass
    class Config(Exporter.Config):
        # models/exporters/mesh_exporter.py of the reference (not vendored here), restated field for field
        fmt: str = "obj-mtl"
        save_name: str = "model"
        save_normal: bool = False
        save_uv: bool = True
        save_texture: bool = True
        texture_size: int = 1024
        texture_format: str = "jpg"
        xatlas_chart_options: dict = field(default_factory=dict)
        xatlas_pack_options: dict = field(default_factory=dict)
        context_type: str = "gl"      # no rasteriser context is needed here; accepted and ignored

    cfg: Config

    def configure(self, geometry, material, background) -> None:
        super().configure(geometry, material, background)
        c = self.cfg
        if c.fmt not in ("obj-mtl", "obj"):
            raise ValueError(f"Unsupported mesh export format: {c.fmt}")
        if dict(c.xatlas_chart_options):
            raise ValueError(f"xatlas_chart_options {sorted(dict(c.xatlas_chart_options))} have no counterpart in the "
                             "dreammat_b200 atlas (uvatlas.py)")
        extra = sorted(set(dict(c.xatlas_pack_options)) - {"padding"})
        if extra:
            raise ValueError(f"xatlas_pack_options {extra} have no counterpart in the dreammat_b200 atlas; only 'padding' is read")
        if c.save_texture and not c.save_uv:
            raise ValueError("save_uv must be True when save_texture is True")
        if not isinstance(geometry, DreamMatMesh) or not isinstance(material, DreamMatMaterial):
            raise TypeError(f"mesh-exporter of dreammat_b200 exports its own geometry and material, got "
                            f"{type(geometry).__name__} / {type(material).__name__}")

    def __call__(self) -> List[ExporterOutput]:
        c = self.cfg
        geo, mat = self.geometry.impl, self.material.impl
        mesh = _T.ExportedMesh(v_pos=geo.v_pos, t_pos_idx=geo.t_pos_idx, v_nrm=geo.v_nrm if c.save_normal else None)
        params = {"mesh": mesh, "save_mat": c.fmt == "obj-mtl", "save_normal": c.save_normal, "save_uv": c.save_uv,
                  "save_vertex_color": False, "map_Kd": None, "map_Ks": None, "map_Bump": None, "map_Pm": None, "map_Pr": None,
                  "map_format": c.texture_format}
        padding = int(dict(c.xatlas_pack_options).get("padding", 2))
        if c.fmt == "obj-mtl" and c.save_texture:
            baked = _T.bake_textures(geo, mat, c.texture_size, padding)
            mesh.v_tex, mesh.t_tex_idx = baked["v_tex"], baked["t_tex_idx"]
            params.update(map_Kd=baked["map_Kd"], map_Pm=baked["map_Pm"], map_Pr=baked["map_Pr"])
        elif c.save_uv:
            from .uvatlas import build_atlas
            atlas = build_atlas(geo.v_pos.numpy(), geo.t_pos_idx.numpy(), c.texture_size, padding)
            mesh.v_tex, mesh.t_tex_idx = torch.from_numpy(atlas.v_tex), torch.from_numpy(atlas.t_tex_idx)
        if c.fmt == "obj" and c.save_texture:
            mesh.v_rgb = _T.vertex_material(geo, mat)[:, :3].cpu()         # per-vertex albedo
            params["save_vertex_color"] = True
        return [ExporterOutput(save_name=f"{c.save_name}.obj", save_type="obj", params=params)]
