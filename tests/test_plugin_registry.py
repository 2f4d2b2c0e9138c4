"""Drop-in boundary (SURVEY.md section 8b), host side, no GPU.

1. The stub `threestudio` package under tests/stub_threestudio (the reference package cannot be imported here:
   pytorch_lightning / omegaconf / nvdiffrast ... are absent) is PINNED against the reference's own code: the event log
   the reference's registry functions and Updateable / BaseObject / BaseModule classes produce for one scenario is
   recorded in tests/golden/threestudio_protocol.json, and the stub must produce the same log.
2. With the stub importable, `import dreammat_b200.threestudio_plugin` must re-register the five names of
   configs/dreammat.yaml:28-97, construct through `cls(cfg)` -> `configure()`, reject unknown config keys, and
   produce / accept the reference's state-dict keys with strict=True.
"""
import dataclasses
import json
import os
import sys
import textwrap

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STUB = os.path.join(ROOT, "tests", "stub_threestudio")
PROTOCOL = os.path.join(ROOT, "tests", "golden", "threestudio_protocol.json")

FIVE = ["dreammat-system", "dreammat-mesh", "dreammat-material", "raytracing-renderer", "stable-diffusion-dreammat-guidance"]

# configs/dreammat.yaml:28-115 (values are the interface; `???` entries filled like cmd/run_examples.sh does)
YAML_GEOMETRY = dict(radius=1.0, shape_init="mesh:PLACEHOLDER", shape_init_params=0.7, shape_init_mesh_up="+y", shape_init_mesh_front="+z",
                     pos_encoding_config=dict(otype="HashGrid", n_levels=16, n_features_per_level=2, log2_hashmap_size=19,
                                              base_resolution=16, per_level_scale=1.447269237440378),
                     n_input_dims=3, n_feature_dims=5)
YAML_GUIDANCE = dict(use_controlnet=True, width=512, height=512, cache_dir="model",
                     pretrained_model_name_or_path="stabilityai/stable-diffusion-2-1-base", controlnet_path="model/controlnet",
                     control_types=["light"], cond_scale=1.05, uncond_scale=[0, -1.0, -0.5, 2000], null_scale=[0, 0.0, -0.5, 2000],
                     noise_scale=0.0, min_step_percent=[500, 0.2, 0.02, 501], max_step_percent=[500, 0.8, 0.5, 501],
                     control_anneal_start_step=700, condition_scales=[1.0], condition_scales_anneal=[0.8])
YAML_MATERIAL = dict(material_activation="sigmoid", environment_texture="load/lights/envmap", environment_scale=2.0, min_metallic=0.0,
                     max_metallic=0.9, min_roughness_squre=0.01, max_roughness_squre=0.9, use_bump=False, use_raytracing=True,
                     diffuse_sample_num=200, specular_sample_num=128)
YAML_SYSTEM = dict(init_step=0, init_width=512, init_height=512, save_train_image=True, save_train_image_iter=1000,
                   geometry_type="dreammat-mesh", geometry=YAML_GEOMETRY, guidance_type="stable-diffusion-dreammat-guidance",
                   guidance=YAML_GUIDANCE, prompt_processor_type="stable-diffusion-prompt-processor",
                   prompt_processor=dict(prompt="a wooden apple"), material_type="dreammat-material", material=YAML_MATERIAL,
                   background_type="solid-color-background", renderer_type="raytracing-renderer", renderer=dict(context_type="cuda"),
                   loggers=dict(wandb=dict(enable=False, project="threestudio")), loss=dict(lambda_sds=1.0, lambda_mat_reg=1.0),
                   optimizer=dict(name="Adam", args=dict(betas=[0.9, 0.99], eps=1e-15, lr=0.01)))


@pytest.fixture()
def stub_on_path():
    for m in [k for k in sys.modules if k == "threestudio" or k.startswith("threestudio.") or k == "dreammat_b200.threestudio_plugin"]:
        del sys.modules[m]
    sys.path.insert(0, STUB)
    try:
        yield
    finally:
        sys.path.remove(STUB)
        for m in [k for k in sys.modules if k == "threestudio" or k.startswith("threestudio.") or k == "dreammat_b200.threestudio_plugin"]:
            del sys.modules[m]


def _scenario(ns):
    """drive registry + construction protocol + Updateable walk; returns an event log"""
    log = []
    register, find = ns["register"], ns["find"]

    @register("x")
    class A:
        pass

    @register("x")
    class B:
        pass
    log.append(("find", find("x").__name__))
    try:
        find("missing")
    except KeyError:
        log.append(("missing", "KeyError"))
    BaseObject, BaseModule, Updateable = ns["BaseObject"], ns["BaseModule"], ns["Updateable"]

    class Child(BaseObject):
        @dataclasses.dataclass
        class Config:
            k: int = 3

        def configure(self, *a, **kw):
            log.append(("child.configure", self.cfg.k, a, tuple(sorted(kw))))

        def update_step(self, epoch, global_step, on_load_weights=False):
            log.append(("child.update", epoch, global_step, on_load_weights))

        def update_step_end(self, epoch, global_step):
            log.append(("child.end", epoch, global_step))

    class Parent(BaseModule):
        @dataclasses.dataclass
        class Config(BaseModule.Config):
            z: float = 1.5

        def configure(self, *a, **kw):
            log.append(("parent.configure", self.cfg.z, self.cfg.weights, a, tuple(sorted(kw))))
            self.child = Child({"k": 7}, 1, two=2)
            self._hidden = Child({})          # underscore attributes are skipped by the walk

        def update_step(self, epoch, global_step, on_load_weights=False):
            log.append(("parent.update", epoch, global_step))

    p = Parent({"z": 2.5}, "pos", kw=1)
    log.append(("device", str(p.device), isinstance(p, Updateable), isinstance(p, torch.nn.Module)))
    log.append(("dummy_in_state_dict", "_dummy" in p.state_dict()))
    p.do_update_step(3, 40)
    p.do_update_step_end(3, 40)
    try:
        Child({"unknown_key": 1})
    except Exception:
        log.append(("unknown", "raises"))
    return log


def test_stub_matches_reference_protocol(stub_on_path):
    """The reference's own register / find / Updateable / BaseObject / BaseModule, driven through `_scenario` with its two
    un-importable helpers injected (parse_structured without omegaconf, get_device as in the stub), produced the log in
    tests/golden/threestudio_protocol.json; the stub must produce the same one."""
    import threestudio as stub
    from threestudio.utils import base as sbase
    from threestudio.utils.misc import get_device
    stub_ns = dict(register=stub.register, find=stub.find, BaseObject=sbase.BaseObject, BaseModule=sbase.BaseModule,
                   Updateable=sbase.Updateable)
    with open(PROTOCOL) as f:
        want = json.load(f)["log"]
    # both sides asked the same injected get_device(): the recorded entry holds no device name
    want = [[e[0], str(get_device()), *e[2:]] if e[0] == "device" else e for e in want]
    a = json.loads(json.dumps(_scenario(stub_ns)))      # tuples -> lists, as recorded
    assert a == want, "\n".join(f"{x}   |   {y}" for x, y in zip(a, want))
    assert ["unknown", "raises"] in a and ["find", "B"] in a


def _write_obj(path):
    from oracle import render as OR          # test infrastructure: a small closed mesh
    v, f = OR.icosphere(2, 0.8, 0.1)
    with open(path, "w") as fh:
        for p in v.tolist():
            fh.write("v %f %f %f\n" % tuple(p))
        for t in f.tolist():
            fh.write("f %d %d %d\n" % (t[0] + 1, t[1] + 1, t[2] + 1))


def _expected_geometry_keys():
    """state-dict keys of the reference's `dreammat-mesh` module (dreammat_mesh.py:126-139 encoding / feature_network /
    three weight-normed predictors, :207-222 mesh buffers; geometry/base.py:199-215 bbox buffers; `_dummy` is
    non-persistent, utils/base.py:113)."""
    keys = ["bbox3d", "bbox2d", "encoding.encoding.encoding.params", "feature_network.layers.0.weight", "feature_network.layers.2.weight"]
    for pred in ("metallic_predictor", "roughness_predictor", "albedo_predictor"):
        for i in (0, 2, 4, 6):
            keys += [f"{pred}.{i}.bias", f"{pred}.{i}.weight_g", f"{pred}.{i}.weight_v"]
    keys += ["v_buffer", "vnrm_buffer", "vtex_buffer", "t_buffer"]
    return keys


def test_plugin_registers_and_constructs_through_the_registry(stub_on_path, tmp_path):
    import threestudio
    before = dict(threestudio.__modules__)
    import dreammat_b200.threestudio_plugin as plug   # noqa: F401
    for name in FIVE:
        assert name in threestudio.__modules__ and name not in before
        assert threestudio.find(name).__module__ == "dreammat_b200.threestudio_plugin"
    from threestudio.utils.base import BaseModule, BaseObject, Updateable
    assert issubclass(threestudio.find("dreammat-mesh"), BaseModule) and issubclass(threestudio.find("raytracing-renderer"), BaseModule)
    assert issubclass(threestudio.find("stable-diffusion-dreammat-guidance"), BaseObject)
    assert issubclass(threestudio.find("stable-diffusion-dreammat-guidance"), Updateable)
    from threestudio.systems.base import BaseLift3DSystem
    assert issubclass(threestudio.find("dreammat-system"), BaseLift3DSystem)

    # ---- geometry through cls(cfg) -> configure(), with the yaml's values
    obj = tmp_path / "apple.obj"
    _write_obj(str(obj))
    gcfg = dict(YAML_GEOMETRY, shape_init=f"mesh:{obj}")
    geo = threestudio.find("dreammat-mesh")(gcfg)
    sd = geo.state_dict()
    assert sorted(sd.keys()) == sorted(_expected_geometry_keys())
    assert sd["encoding.encoding.encoding.params"].shape == (12599920,) and sd["feature_network.layers.0.weight"].shape == (64, 32)
    assert sd["feature_network.layers.2.weight"].shape == (5, 64) and sd["metallic_predictor.0.weight_v"].shape == (256, 63)
    assert sd["albedo_predictor.6.weight_g"].shape == (3, 1) and sd["t_buffer"].dtype == torch.int64
    trainable = [n for n, p in geo.named_parameters() if p.requires_grad]
    assert trainable == ["encoding.encoding.encoding.params", "feature_network.layers.0.weight", "feature_network.layers.2.weight"]
    # the three parameters are views of the implementation's ONE flat buffer (what the fused Adam / all-reduce use)
    impl = geo.impl
    assert sd["encoding.encoding.encoding.params"].data_ptr() == impl.params.data_ptr()
    geo.feature_network.layers[2].weight.data.fill_(0.25)
    assert float(impl.params[-1]) == 0.25
    # strict round trip, as a reference-written checkpoint would be loaded (systems/base.py:52-58)
    sd2 = {k: (torch.randn_like(v) if v.is_floating_point() else v.clone()) for k, v in sd.items()}
    geo.load_state_dict(sd2, strict=True)
    assert torch.equal(impl.params[:impl.n_grid], sd2["encoding.encoding.encoding.params"])
    assert torch.equal(impl.W2, sd2["feature_network.layers.2.weight"])
    mesh = geo.isosurface()
    assert mesh.v_pos.shape[1] == 3 and mesh.t_pos_idx.shape[1] == 3 and float(mesh.v_pos.abs().max()) == pytest.approx(0.7, rel=1e-6)
    # ---- config errors behave like the reference's
    with pytest.raises(Exception):
        threestudio.find("dreammat-mesh")(dict(gcfg, not_a_field=1))                       # unknown key (OmegaConf error there)
    with pytest.raises(ValueError, match="does not exist"):
        threestudio.find("dreammat-mesh")(dict(gcfg, shape_init="mesh:/nonexistent.obj"))   # dreammat_mesh.py:145-146
    with pytest.raises(ValueError, match="Unknown shape initialization"):
        threestudio.find("dreammat-mesh")(dict(gcfg, shape_init="sphere"))                  # :224-227
    # ---- every key of the yaml's guidance / material / system blocks is a Config field with the reference's default
    G = threestudio.find("stable-diffusion-dreammat-guidance").Config(**YAML_GUIDANCE)
    assert G.half_precision_weights is True and G.view_dependent_prompting is True and G.condition_scales_anneal == [0.8]
    M = threestudio.find("dreammat-material").Config(**YAML_MATERIAL)
    assert M.min_roughness == 0.1 and M.geometry_type == "schlick" and M.weights is None
    S = threestudio.find("dreammat-system").Config(**YAML_SYSTEM)
    assert S.texture is True and S.exporter_type == "mesh-exporter" and S.latent_steps == 1000
    with pytest.raises(FileNotFoundError):    # weights come from local diffusers-format directories only; absent -> loud
        threestudio.find("stable-diffusion-dreammat-guidance")(dict(YAML_GUIDANCE, cache_dir=str(tmp_path)))


def test_vae_legacy_attention_keys_and_config_json(tmp_path):
    """ADVICE r1: published AutoencoderKL checkpoints use query/key/value/proj_attn (some as 1x1 convs); config.json drives
    the architecture."""
    import json
    from dreammat_b200 import weights as W
    w = {"encoder.mid_block.attentions.0.query.weight": torch.randn(8, 8, 1, 1), "encoder.mid_block.attentions.0.query.bias": torch.randn(8),
         "encoder.mid_block.attentions.0.key.weight": torch.randn(8, 8), "encoder.mid_block.attentions.0.value.weight": torch.randn(8, 8),
         "encoder.mid_block.attentions.0.proj_attn.weight": torch.randn(8, 8, 1, 1), "encoder.mid_block.attentions.0.group_norm.weight": torch.randn(8),
         "encoder.conv_in.weight": torch.randn(8, 3, 3, 3)}
    n = W.normalize_vae_keys(w)
    p = "encoder.mid_block.attentions.0."
    assert set(n) == {p + "to_q.weight", p + "to_q.bias", p + "to_k.weight", p + "to_v.weight", p + "to_out.0.weight", p + "group_norm.weight",
                      "encoder.conv_in.weight"}
    assert n[p + "to_q.weight"].shape == (8, 8) and n[p + "to_out.0.weight"].shape == (8, 8) and n["encoder.conv_in.weight"].shape == (8, 3, 3, 3)
    assert torch.equal(n[p + "to_q.weight"], w[p + "query.weight"].reshape(8, 8))
    assert W.normalize_vae_keys(n).keys() == n.keys()                     # idempotent on current names
    (tmp_path / "u.json").write_text(json.dumps({"attention_head_dim": [5, 10, 20, 20], "block_out_channels": [320, 640, 1280, 1280],
                                                 "cross_attention_dim": 1024, "layers_per_block": 2, "norm_num_groups": 32}))
    (tmp_path / "c.json").write_text(json.dumps({"conditioning_embedding_out_channels": [16, 32, 96, 256], "conditioning_channels": 22}))
    assert W.unet_config_from_json(str(tmp_path / "u.json"), str(tmp_path / "c.json")) == W.UNetConfig()
    (tmp_path / "v.json").write_text(json.dumps({"block_out_channels": [128, 256, 512, 512], "latent_channels": 4, "scaling_factor": 0.18215}))
    assert W.vae_config_from_json(str(tmp_path / "v.json")) == W.VAEConfig()
    assert W.unet_config_from_json("/nonexistent") == W.UNetConfig()


def test_training_step_host_logic_matches_reference_execution(stub_on_path):
    """The plugin system's training_step against a record of the reference's own `DreamMat.training_step`
    (systems/dreammat.py:57-179) executed with recording stand-ins (tests/golden/make_system_golden.py): what the guidance is
    handed, the loss assembly with scheduled weights, the names / order / values of everything logged, and the train-image grid.
    Both branches: op-by-op (`fused_step=False`) and fused (the kernel sequence stood in by a stub returning the same numbers)."""
    import types

    import dreammat_b200.threestudio_plugin as P
    from dreammat_b200.guidance import C
    from tests.golden.make_system_golden import scenario
    G = torch.load(os.path.join(ROOT, "tests", "golden", "system_vectors.pt"))
    for rec in G["records"]:
        step = rec["step"]
        for fused in (False, True):
            out, gout, batch = scenario(step)
            log, grids, seen = [], [], {}

            class Sys:
                cfg = types.SimpleNamespace(loss=dict(G["loss_cfg"]), save_train_image=True, save_train_image_iter=rec["save_iter"],
                                            texture=True, fused_step=fused)
                true_global_step, true_current_epoch = step, 0
                training_step, _log, _save_train_images = P.DreamMat.training_step, P.DreamMat._log, P.DreamMat._save_train_images

                def __call__(self, b):
                    seen["renderer_batch_keys"] = sorted(b)
                    return out

                def prompt_processor(self):
                    return "PROMPT_UTILS"

                def log(self, name, value):
                    log.append((name, float(value)))

                def C(self, v):
                    return C(v, self.true_current_epoch, self.true_global_step)

                def guidance(self, rgb, prompt_utils, **kw):
                    seen["guidance"] = dict(rgb_is_comp_rgb=rgb is out["comp_rgb"], prompt_utils=prompt_utils, keys=sorted(kw),
                                            cond_normal_is_comp_normal=kw.get("cond_normal") is out["comp_normal"],
                                            cond_depth_is_comp_depth=kw.get("cond_depth") is out["comp_depth"], rgb_as_latents=kw.get("rgb_as_latents"))
                    return dict(gout, _grad=torch.zeros(1))        # the product's guidance also returns private `_` entries: never logged

                def save_image_grid(self, fn, imgs=None, name=None, step=None):
                    grids.append(dict(filename=fn, name=name, step=step, rows=imgs))
            me = Sys()
            if fused:
                lam = {k: C(v, 0, step) for k, v in G["loss_cfg"].items()}
                flat = torch.zeros(6, requires_grad=True)

                class Impl:        # stands for system.DreamMat: same numbers as the op-by-op branch would produce
                    def training_step_fused(self, b, apply_optimizer=True):
                        assert apply_optimizer is False
                        return {"loss": lam["lambda_sds"] * gout["loss_sds"] + lam["lambda_mat_reg"] * out["loss_mat_reg"], "loss_sds": gout["loss_sds"],
                                "loss_mat_reg": out["loss_mat_reg"], "comp_rgb": out["comp_rgb"], **{k: v for k, v in gout.items() if k.endswith("_norm")}}
                me.impl = Impl()
                layers = [types.SimpleNamespace(weight=flat[2:4]), None, types.SimpleNamespace(weight=flat[4:6])]
                me.geometry = types.SimpleNamespace(impl=types.SimpleNamespace(dgrid=torch.ones(2), dW1=torch.ones(2), dW2=torch.ones(2)),
                                                    encoding=types.SimpleNamespace(encoding=types.SimpleNamespace(encoding=types.SimpleNamespace(params=flat[0:2]))),
                                                    feature_network=types.SimpleNamespace(layers=layers))
            ret = me.training_step(dict(batch), 0)
            assert abs(float(ret["loss"]) - rec["loss"]) < 1e-5 * max(1.0, abs(rec["loss"])), (step, fused, float(ret["loss"]), rec["loss"])
            want = dict(rec["log"])
            got = dict(log)
            assert set(got) == set(want), (step, fused, sorted(set(got) ^ set(want)))
            for k, v in want.items():
                assert abs(got[k] - v) < 1e-5 * max(1.0, abs(v)), (k, got[k], v)
            if not fused:
                assert [n for n, _ in log] == [n for n, _ in rec["log"]]                      # same order, too
                assert seen == rec["seen"]
            else:
                ret["loss"].backward()                                                     # the carried gradient reaches the leaves
                assert torch.equal(flat.grad, torch.ones(6))
            assert len(grids) == len(rec["grids"])
            for ours, ref in zip(grids, rec["grids"]):
                assert (ours["filename"], ours["name"], ours["step"]) == (ref["filename"], ref["name"], ref["step"])
                assert [len(r) for r in ours["rows"]] == [len(r) for r in ref["rows"]] == [8, 8]
                for ro, rr in zip(ours["rows"], ref["rows"]):
                    for co, cr in zip(ro, rr):
                        assert co["type"] == cr["type"] and co["kwargs"] == cr["kwargs"] and torch.equal(co["img"], cr["img"])


def test_validation_and_test_hooks_match_reference_execution(stub_on_path):
    """validation_step / test_step / on_test_epoch_end of the plugin system against a record of the reference's own hooks
    (systems/dreammat.py:181-300): file names, grid layouts with and without `texture`, the four RGBA maps per test view
    (albedo / roughness / metallic / render over the opacity), the turntable gif."""
    import types

    import dreammat_b200.threestudio_plugin as P
    from tests.golden.make_system_golden import scenario
    G = torch.load(os.path.join(ROOT, "tests", "golden", "system_vectors.pt"))
    assert [e["texture"] for e in G["evals"]] == [True, False]
    for ev in G["evals"]:
        out, _, batch = scenario(77)
        batch["index"] = torch.tensor([7])
        calls = []

        class Sys:
            cfg = types.SimpleNamespace(texture=ev["texture"])
            true_global_step = 1234
            validation_step, test_step, on_test_epoch_end = P.DreamMat.validation_step, P.DreamMat.test_step, P.DreamMat.on_test_epoch_end
            _grid, _cell = P.DreamMat._grid, staticmethod(P.DreamMat._cell)

            def __call__(self, b):
                return out

            def save_image_grid(self, fn, imgs=None, name=None, step=None):
                calls.append(("grid", fn, name, step, imgs))

            def save_img(self, img, fn):
                calls.append(("img", fn, img))

            def save_gif(self, path, fps=None):
                calls.append(("gif", path, fps))
        me = Sys()
        me.validation_step(batch)
        me.test_step(batch)
        me.on_test_epoch_end()
        assert len(calls) == len(ev["calls"]) == 7
        for ours, ref in zip(calls, ev["calls"]):
            assert ours[0] == ref[0] and ours[1] == ref[1], (ours[:2], ref[:2])
            if ours[0] == "grid":
                assert ours[2:4] == ref[2:4] and len(ours[4]) == len(ref[4])
                for co, cr in zip(ours[4], ref[4]):
                    assert co["type"] == cr["type"] and co["kwargs"] == cr["kwargs"] and torch.equal(co["img"], cr["img"])
            elif ours[0] == "img":
                assert ours[2].shape[-1] == 4 and torch.equal(ours[2], ref[2])
            else:
                assert ours[2] == ref[2] == 30
