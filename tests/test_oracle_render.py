"""CPU checks that pin the render-side oracle (no GPU, runs in seconds)."""
import math
import os

import numpy as np
import torch

from oracle import render as O
from tests._fixtures import make_scene, rel_err

ASSETS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "splitsum_assets.pt")


def test_bvh_matches_brute_force():
    v, f = O.icosphere(2, radius=0.8, bump=0.15)
    g = torch.Generator().manual_seed(1)
    ro = torch.randn(4000, 3, generator=g) * 0.6
    rd = torch.nn.functional.normalize(torch.randn(4000, 3, generator=g), dim=-1)
    t0, i0, uv0 = O.RayTracer(v.numpy(), f.numpy(), brute=True).trace_raw(ro.numpy(), rd.numpy())
    t1, i1, uv1 = O.RayTracer(v.numpy(), f.numpy()).trace_raw(ro.numpy(), rd.numpy())
    assert (i0 == i1).all()
    assert np.array_equal(t0, t1)
    assert np.array_equal(uv0, uv1)
    assert (i0 >= 0).sum() > 1000 and (i0 < 0).sum() > 100


def test_hashgrid_layout_matches_survey():
    meta, total = O.hashgrid_meta()
    assert [m["size"] for m in meta[:6]] == [4096, 13824, 39304, 117656, 357912, 524288]
    assert total * 2 == 12599920  # geometry.encoding.encoding.encoding.params (SURVEY.md section 5)
    assert [m["hashed"] for m in meta[:6]] == [False] * 5 + [True]


def test_hashgrid_is_trilinear_and_differentiable():
    meta, total = O.hashgrid_meta()
    p = (torch.rand(total * 2, dtype=torch.float64) * 2e-4 - 1e-4).requires_grad_(True)
    x = torch.rand(5, 3, dtype=torch.float64)
    enc = O.hashgrid_encode(x, p, meta)
    assert enc.shape == (5, 32)
    (g,) = torch.autograd.grad(enc.sum(), p)
    # each point touches <= 8 corners x 16 levels x 2 features, weights sum to 1 per level/feature
    assert abs(float(g.sum()) - 5 * 32) < 1e-9


def test_direction_tables():
    t = O.direction_tables(200)
    assert t.shape == (200, 2) and float(t.min()) >= 0 and float(t.max()) <= 1
    # k = N..2N-1 -> z in [0,1): upper hemisphere only; ue = 1 - 2 asin(z)/pi
    assert abs(float(t[0, 1]) - 1.0) < 1e-6


def test_mc_shading_white_furnace_and_grad():
    sc = make_scene(res=24, subdiv=2, bump=0.0)
    pn = sc["pn"]
    env = torch.ones(64, 128, 3)
    f = sc["features"].clone().requires_grad_(True)
    albedo, metallic, rough, reg = O.material_params(f, sc["features_jitter"])
    out = O.shade_raytracing(sc["pts"], sc["nrm"], sc["vd"], env, metallic, rough, albedo, sc["rand_d"], sc["rand_s"],
                             lambda o, d: sc["tracer"].trace(o, d)[1])
    # convex sphere under a constant white map: every diffuse sample sees L=1 -> diffuse colour = albedo
    dl = out["diffuse_lights"]
    assert float((dl - 1.0).abs().max()) < 0.03  # the horizon sample may graze the faceted surface
    (g,) = torch.autograd.grad(out["color"].sum() + reg, f)
    assert torch.isfinite(g).all() and float(g.abs().sum()) > 0


def test_fg_lut_fixture_is_the_split_sum_brdf_integral():
    """Pins fg_lookup's axis convention (u = N.V -> W, v = roughness -> H) against the only golden
    data the reference holds for this path: the LUT must equal Karis' split-sum DFG integral.
    The reference's load/lights/bsdf_256_256.bin is stored whole in tests/golden/splitsum_assets.pt."""
    lut = torch.load(ASSETS)["fg_lut"][0]

    def dfg(ndv, rough, n=4096):
        a = rough * rough
        i = torch.arange(n, dtype=torch.float64)
        u1 = (i + 0.5) / n
        # radical inverse base 2
        bits = i.long()
        ri = torch.zeros(n, dtype=torch.float64)
        fct = 0.5
        for _ in range(32):
            ri += (bits & 1).double() * fct
            bits >>= 1
            fct *= 0.5
        phi = 2 * math.pi * u1
        ct = torch.sqrt((1 - ri) / (1 + (a * a - 1) * ri))
        st = torch.sqrt(1 - ct * ct)
        H = torch.stack([st * torch.cos(phi), st * torch.sin(phi), ct], -1)
        V = torch.tensor([math.sqrt(1 - ndv * ndv), 0.0, ndv], dtype=torch.float64)
        VoH = (H * V).sum(-1)
        L = 2 * VoH[:, None] * H - V
        NoL, NoH = L[:, 2].clamp(min=0), H[:, 2].clamp(min=0)
        VoH = VoH.clamp(min=0)
        # height-correlated Smith GGX visibility (what the shipped LUT was baked with)
        lv = NoL * math.sqrt(ndv * ndv * (1 - a * a) + a * a)
        ll = ndv * torch.sqrt(NoL * NoL * (1 - a * a) + a * a)
        G = 2 * NoL * ndv / (lv + ll + 1e-12)
        Gv = G * VoH / (NoH * ndv + 1e-12)
        Fc = (1 - VoH) ** 5
        m = NoL > 0
        return float(((1 - Fc) * Gv)[m].sum() / n), float((Fc * Gv)[m].sum() / n)

    for ndv, rough in ((0.5, 0.5), (0.8, 0.3), (0.3, 0.8), (0.2, 0.9)):
        got = O.fg_lookup(lut, torch.tensor([ndv]), torch.tensor([rough]))[0]
        want = dfg(ndv, rough)
        assert abs(float(got[0]) - want[0]) < 0.01 and abs(float(got[1]) - want[1]) < 0.004, (ndv, rough, got, want)
    # spot values recorded in SURVEY.md section 8c
    assert abs(float(lut[0, 0, 0]) - 0.00973) < 1e-4 and abs(float(lut[128, 128, 0]) - 0.83426) < 1e-4


def test_envlight_white_furnace():
    env = torch.ones(32, 64, 3) * 0.5
    diffuse, spec = O.build_envlight(env, scale=2.0, max_res=32, min_res=16)
    assert len(spec) == 2
    assert float((diffuse - 1.0).abs().max()) < 2e-2  # cosine integral of a constant (cos clamped at .999)
    for m in spec:
        assert float((m - 1.0).abs().max()) < 1e-4
    d = torch.nn.functional.normalize(torch.randn(64, 3), dim=-1)
    assert float((O.cube_sample_linear(spec[0], d) - 1.0).abs().max()) < 1e-4


def test_cube_sampling_is_continuous_across_faces():
    g = torch.Generator().manual_seed(0)
    cube = O.latlong_to_cubemap(O.synthetic_envmap(64, 128), 16)
    d = torch.nn.functional.normalize(torch.randn(2000, 3, generator=g), dim=-1)
    e = torch.nn.functional.normalize(d + 1e-4 * torch.randn(2000, 3, generator=g), dim=-1)
    a, b = O.cube_sample_linear(cube, d), O.cube_sample_linear(cube, e)
    assert float((a - b).abs().max()) < 0.05 * float(cube.max())


def test_gbuffer_and_jitter_shapes():
    sc = make_scene(res=32, subdiv=2)
    gb = sc["gb"]
    assert gb["rast"].shape == (1, 32, 32, 4)
    cov = gb["selector"].float().mean()
    assert 0.05 < float(cov) < 0.9
    # interpolated position lies on the pixel-centre ray
    o = sc["cam"]["rays_o"].reshape(-1, 3)[gb["selector"][0]]
    d = sc["cam"]["rays_d"].reshape(-1, 3)[gb["selector"][0]]
    t = ((sc["pts"] - o) * d).sum(-1, keepdim=True)
    assert float((o + t * d - sc["pts"]).abs().max()) < 1e-4
    pj = O.jitter_positions(sc["pts"], sc["nrm"], sc["rand_ang"], sc["normal_eps"])
    off = pj - sc["pts"]
    assert float((off * sc["nrm"]).sum(-1).abs().max()) < 1e-5  # stays in the tangent plane


def test_antialias_pairs_product_host_code_matches_oracle():
    """The cached silhouette-blend list (dreammat_b200/antialias.py, vectorised numpy, init-time host code) against the
    oracle's scalar restatement; and the blend is a partition-of-unity operation."""
    from dreammat_b200 import antialias as A
    sc = make_scene(res=40, subdiv=2, bump=0.15, seed=1, n_views=2)
    nbr = A.edge_neighbours(sc["f"].numpy().astype(np.int64), sc["v"].shape[0])
    assert (nbr >= 0).all()          # closed mesh: every edge has a neighbour
    for b in range(2):
        rast = sc["gb"]["rast"][b]
        pairs = O.antialias_pairs(rast, sc["v"], sc["f"], sc["cam"]["mvp_mtx"][b])
        d, s, a = A.build_pairs(rast.numpy(), sc["v"].numpy(), sc["f"].numpy().astype(np.int64), nbr,
                                sc["cam"]["mvp_mtx"][b].numpy())
        po = sorted((p[0], p[1], round(p[2], 4)) for p in pairs)
        pp = sorted((int(x), int(y), round(float(z), 4)) for x, y, z in zip(d, s, a))
        assert po == pp and len(po) > 20
        assert 0 < min(p[2] for p in pairs) and max(p[2] for p in pairs) <= 0.5
        x = torch.full((40 * 40, 3), 0.7)
        assert float((O.antialias_apply(x, pairs) - x).abs().max()) < 1e-6   # constant images are fixed points
        # the mask gets fractional coverage on both sides of the silhouette
        m = sc["gb"]["mask"][b].reshape(-1, 1).float()
        ma = O.antialias_apply(m, pairs)
        assert ((ma > 0.01) & (ma < 0.99)).sum() > 20
