"""Prior extraction from camera rays: the fused density level of the main field (ps_density_level_fwd / _ms, the
proposal kernels instantiated for the field's density head), `get_surface_hits`, ps_surface_hits and `PriorExtractor`,
against the stand-alone kernel chain, `get_depth`, the reference fixture and the public pieces composed by hand."""
import ctypes as C
import dataclasses
import pickle

import pytest
import torch

from helpers import Fixture
from oracle.priors_oracle import read_priors_like_city_prior
from test_gpu_model import build_model, make_field

pytestmark = pytest.mark.gpu
DEV = "cuda"
AABB = [-1.0, -1.0, -0.5, 1.0, 1.0, 0.5]


def rel_l2(a, b):
    a, b = a.double(), b.double()
    return float((a - b).norm() / (b.norm() + 1e-30))


def random_field(L, F, seed=0, log2T=14):
    from presight_b200.field_components.spatial_distortions import SceneContraction
    from presight_b200.fields.ingp_field import iNGPField
    torch.manual_seed(seed)
    f = iNGPField(torch.tensor([AABB[:3], AABB[3:]]), hidden_dim=64, num_levels=L, max_res=2048, base_res=16,
                  features_per_level=F, log2_hashmap_size=log2T, spatial_distortion=SceneContraction(order=float("inf")),
                  use_semantics=True, semantic_dim=64, appearance_embedding_dim=16, implementation="b200")
    with torch.no_grad():
        f.mlp_base_grid.hash_table.mul_(300.0)       # init-scale tables give a featureless field
    return f.to(DEV)


def rays(n, S, seed=0):
    g = torch.Generator().manual_seed(seed)
    o = ((torch.rand(n, 3, generator=g) - 0.5) * torch.tensor([1.0, 1.0, 0.1])).to(DEV)
    d = torch.nn.functional.normalize(torch.randn(n, 3, generator=g), dim=-1).to(DEV)
    eu = (torch.rand(n, S + 1, generator=g) * 0.05 + 0.001).cumsum(-1).to(DEV)
    return o, d, eu


def kernel_weights(field, o, d, eu):
    from presight_b200 import fused
    from presight_b200._lib import call, host_floats, host_prop_net, ptr, stream
    l0, l1 = list(field.mlp_base_mlp.layers)
    g = field._grid_meta()
    N, S = eu.shape[0], eu.shape[1] - 1
    w = torch.empty(N, S, device=DEV)
    net = host_prop_net([l0.weight.detach(), l1.weight.detach()], [l0.bias.detach(), l1.bias.detach()])
    call("ps_density_level_fwd", C.byref(net), ptr(o), ptr(d), ptr(eu), N, S, host_floats(field.aabb_host()), 1,
         ptr(field.mlp_base_grid.hash_table.detach()), host_floats(g.scalings), g.L, g.F, g.log2_T, ptr(w), stream())
    assert fused.tc5_density_supported(g, 64, field.mlp_base_mlp.precision, S)
    return w


def chain_weights(density_fn, o, d, eu):
    """ops.get_weights(density_fn(positions)) on the stand-alone kernels (the path get_depth takes)."""
    from presight_b200 import ops
    from presight_b200.cameras.rays import RayBundle
    rs = RayBundle(origins=o, directions=d).get_ray_samples(eu[:, :-1, None], eu[:, 1:, None])
    density = density_fn(rs.frustums.get_positions())
    return ops.get_weights((eu[:, 1:] - eu[:, :-1])[..., None].contiguous(), density.contiguous())[..., 0]


@pytest.mark.parametrize("case,S", [("L16F2", 64), ("L10F4", 64), ("L10F4", 128), ("fixture", 32), ("L16F2", 96)])
def test_density_level_weights_match_standalone_chain(case, S):
    if case == "fixture":
        fx = Fixture("fields.npz")
        field = make_field(fx, fx.sub("field/"), "b200")          # L6 F2: the K0 = 16 instantiation
    else:
        field = random_field(int(case[1:3]), int(case[-1]))
    o, d, eu = rays(1500, S, seed=S)
    with torch.no_grad():
        got = kernel_weights(field, o, d, eu)
        want = chain_weights(lambda p: field.density_fn(p)[0], o, d, eu)
    assert torch.isfinite(got).all()
    assert want.abs().max() > 1e-3, "featureless field"
    assert rel_l2(got, want) <= 1e-2, rel_l2(got, want)


def presight_model(log2T=14, S_final=64, nf=16, impl="b200"):
    from presight_b200 import synthetic
    from presight_b200.model import NerfactoNuscMSModel
    cfg = synthetic.config_presight(impl)
    cfg = dataclasses.replace(cfg, log2_hashmap_size=log2T, num_nerf_samples_per_ray=S_final,
                              proposal_net_args_list=[dict(a, log2_hashmap_size=log2T) for a in cfg.proposal_net_args_list])
    torch.manual_seed(2)
    if nf == 1:
        cen, aabbs = torch.zeros(1, 3), synthetic.tile_aabb()
    else:
        cen, aabbs = synthetic.sub_field_layout(nf)
    model = NerfactoNuscMSModel(cfg, cen, aabbs)
    with torch.no_grad():
        for f in model.field.fields:
            f.mlp_base_grid.hash_table.mul_(300.0)
        for p in model.proposal_networks:
            for f in p.fields:
                f.encoding.hash_table.mul_(300.0)
    return model.to(DEV).eval(), cfg


def c2_model(S_final=64, impl="b200", log2T=14):
    from presight_b200 import synthetic
    cfg = synthetic.config_c2(impl)
    cfg = dataclasses.replace(cfg, log2_hashmap_size=log2T, num_nerf_samples_per_ray=S_final,
                              proposal_net_args_list=[dict(a, log2_hashmap_size=log2T) for a in cfg.proposal_net_args_list])
    from presight_b200.model import NerfactoNuscMSModel
    torch.manual_seed(4)
    model = NerfactoNuscMSModel(cfg, torch.zeros(1, 3), synthetic.tile_aabb())
    with torch.no_grad():
        for name, p in model.named_parameters():
            if name.endswith("hash_table"):
                p.mul_(300.0)
    return model.to(DEV).eval(), cfg


def synth_bundle(n, seed=5):
    from presight_b200 import synthetic
    from presight_b200.cameras.rays import RayBundle
    host = synthetic.make_rays(n, seed=seed)
    return RayBundle(origins=host["origins"].to(DEV), directions=host["directions"].to(DEV))


def test_routed_density_matches_dispatch_path():
    """16 sub-fields: ps_density_level_fwd_ms on routed points against iNGPFieldMS.density_fn (argsort + per-sub-field
    launch chains)."""
    from presight_b200 import fused
    from presight_b200._lib import PropNetDev, call, device_ptr_array, device_struct_array, host_floats, ptr, stream
    model, _ = presight_model()
    fms = model.field
    rb = synth_bundle(4000)
    g = torch.Generator().manual_seed(3)
    t = (torch.rand(4000, 16, generator=g) * 2.0).to(DEV)               # 0 .. 40 m along the rays (scene units)
    pts = (rb.origins[:, None, :] + rb.directions[:, None, :] * t[..., None]).reshape(-1, 3).contiguous()
    grid = fms.fields[0]._grid_meta()
    with torch.no_grad():
        rt = fused.route_points(fms.centroids, fms._aabbs_host(), True, None, None, None, positions=pts)
        subs = [(f.mlp_base_grid.hash_table, *[x for l in f.mlp_base_mlp.layers for x in (l.weight, l.bias)])
                for f in fms.fields]
        tables = device_ptr_array([s[0] for s in subs], DEV, ("test_density", "tables"))
        nets = device_struct_array([PropNetDev(s[1].data_ptr(), s[2].data_ptr(), s[3].data_ptr(), s[4].data_ptr(),
                                               0, 0, 0, 0) for s in subs], DEV, ("test_density", "nets"))
        got = torch.zeros(pts.shape[0], device=DEV)
        call("ps_density_level_fwd_ms", ptr(nets), 64, ptr(rt.x01), ptr(rt.sel), ptr(rt.perm), ptr(rt.tile_sf), rt.rows,
             ptr(tables), host_floats(grid.scalings), grid.L, grid.F, grid.log2_T, ptr(got), stream())
        want = fms.density_fn(pts)[0].view(-1)
    assert int((rt.sf.long().bincount(minlength=16) > 0).sum()) >= 4, "points reach several sub-fields"
    assert want.abs().max() > 1e-3
    assert rel_l2(got, want) <= 1e-2, rel_l2(got, want)


def test_routed_mode_with_one_sub_field_matches_ray_mode():
    from presight_b200 import fused
    field = random_field(10, 4, seed=6)
    o, d, eu = rays(3000, 64, seed=7)
    l0, l1 = list(field.mlp_base_mlp.layers)
    with torch.no_grad():
        w_ray = kernel_weights(field, o, d, eu)
        d_ray = fused.density_level_depth(o, d, eu, field.mlp_base_grid.hash_table, field.aabb_host(), True,
                                          field._grid_meta(), l0.weight, l0.bias, l1.weight, l1.bias, 0.5)
        params = [(field.mlp_base_grid.hash_table, l0.weight, l0.bias, l1.weight, l1.bias)]
        d_ms = fused.density_level_depth_ms(o, d, eu, torch.zeros(1, 3, device=DEV), [field.aabb_host()], True,
                                            field._grid_meta(), params, 0.5)
        # the routed kernel's densities composited by ps_composite_fwd give the ray kernel's weights
        from presight_b200._lib import PropNetDev, call, device_ptr_array, device_struct_array, host_floats, ptr, stream
        rt = fused.route_points(torch.zeros(1, 3, device=DEV), [field.aabb_host()], True, o, d, eu)
        g = field._grid_meta()
        tables = device_ptr_array([params[0][0]], DEV, ("test_density1", "tables"))
        nets = device_struct_array([PropNetDev(*[t.data_ptr() for t in params[0][1:]], 0, 0, 0, 0)], DEV,
                                   ("test_density1", "nets"))
        den = torch.zeros(o.shape[0] * 64, device=DEV)
        call("ps_density_level_fwd_ms", ptr(nets), 64, ptr(rt.x01), ptr(rt.sel), ptr(rt.perm), ptr(rt.tile_sf), rt.rows,
             ptr(tables), host_floats(g.scalings), g.L, g.F, g.log2_T, ptr(den), stream())
        w_ms = torch.empty_like(w_ray)
        call("ps_composite_fwd", ptr(eu), ptr(den), None, None, o.shape[0], 64, 0, 0.5, ptr(w_ms), None, None, None,
             None, None, None, stream())
    assert float((w_ms - w_ray).abs().max()) <= 1e-6
    assert float((d_ms == d_ray).float().mean()) >= 0.999


@pytest.mark.parametrize("shape", ["c2", "presight16"])
def test_surface_hits_match_get_depth(shape):
    model, _ = c2_model() if shape == "c2" else presight_model()
    assert model.field.supports_level_depth(64)
    rb = synth_bundle(8192, seed=11)
    from presight_b200.cameras.rays import RayBundle
    with torch.no_grad():
        want = model.get_depth(RayBundle(origins=rb.origins, directions=rb.directions))["depth"]
        got = model.get_surface_hits(RayBundle(origins=rb.origins, directions=rb.directions))["depth"]
    assert got.shape == want.shape == (8192, 1)
    close = (got - want).abs() <= 1e-4 * want.abs().max()
    assert float(close.float().mean()) >= 0.99, float(close.float().mean())
    assert rel_l2(got, want) <= 1e-2


def test_surface_hits_against_reference_fixture():
    from presight_b200.cameras.rays import RayBundle
    fx = Fixture("model.npz")
    model = build_model(fx, "b200")
    model.eval()
    with torch.no_grad():
        got = model.get_surface_hits(RayBundle(origins=fx["origins"].to(DEV), directions=fx["dirs"].to(DEV)))["depth"]
    want = fx["depth_eval/depth"]
    assert ((got.cpu() - want).abs() <= 1e-4 * want.abs().max()).float().mean() >= 0.95


@pytest.mark.parametrize("impl,S", [("b200+fp32", 64), ("b200", 48)])
def test_fallback_is_get_depth_bit_for_bit(impl, S):
    from presight_b200.cameras.rays import RayBundle
    model, _ = c2_model(S_final=S, impl=impl)
    assert not model.field.supports_level_depth(S)
    rb = synth_bundle(3000, seed=12)
    with torch.no_grad():
        want = model.get_depth(RayBundle(origins=rb.origins, directions=rb.directions))["depth"]
        got = model.get_surface_hits(RayBundle(origins=rb.origins, directions=rb.directions))["depth"]
    assert torch.equal(got, want)


def run_extractor(model, rb, chunk, **kw):
    from presight_b200.extract import PriorExtractor
    ex = PriorExtractor(model, 0.05, chunk_rays=chunk, **kw)
    ex.add(rb)
    assert ex.n_hits > 0
    return ex.finalize()


def test_extractor_chunking_and_hand_composition():
    from presight_b200 import priors
    from presight_b200.cameras.rays import RayBundle
    from presight_b200.extract import surface_hits
    model, _ = c2_model()
    n = 20000
    rb = synth_bundle(n, seed=13)
    kw = dict(max_range_m=60.0, z_range_m=(-3.0, 12.0))
    one = run_extractor(model, rb, n, **kw)
    five = run_extractor(model, rb, (n + 4) // 5, **kw)
    assert one["n_voxels"] == five["n_voxels"]
    assert torch.equal(one["hits"], five["hits"])
    assert torch.equal(one["features"], five["features"])
    assert float((one["points"] - five["points"]).abs().max()) <= 1e-6
    # the public pieces composed by hand
    with torch.no_grad():
        depth = model.get_surface_hits(RayBundle(origins=rb.origins, directions=rb.directions))["depth"]
        ps, pm, keep = surface_hits(rb.origins, rb.directions, depth, 0.05, **kw)
        dens, feats = model.query_priors(ps)
        k = keep & (dens > 1)
        ref = priors.postprocess_priors(pm[k], feats[k], torch.zeros(int(k.sum()), 3, device=DEV), None)
    assert ref["n_voxels"] == one["n_voxels"]
    assert torch.equal(ref["hits"], one["hits"])
    assert torch.equal(ref["features"], one["features"])
    assert float((ref["points"] - one["points"]).abs().max()) <= 1e-6
    # the metric points the extractor voxelises are ps_surface_hits' own, bit for bit
    from presight_b200.extract import PriorExtractor
    ex = PriorExtractor(model, 0.05, chunk_rays=n, **kw)
    ex.add(rb)
    assert torch.equal(torch.cat(ex._points) / torch.full((1, 3), 0.05, device=DEV), pm[k])
    # the selector drops hits: a looser window keeps more
    assert int(k.sum()) < int((dens > 1).sum())


def test_extractor_with_sub_fields_writes_a_readable_pickle(tmp_path):
    from presight_b200 import priors
    model, _ = presight_model()
    rb = synth_bundle(30000, seed=17)
    colors = torch.rand(30000, 3, generator=torch.Generator().manual_seed(1)).to(DEV)
    from presight_b200.extract import PriorExtractor
    ex = PriorExtractor(model, 0.05, max_range_m=80.0, z_range_m=(None, 15.0), chunk_rays=1 << 13)
    ex.add(rb, colors)
    res = ex.finalize()
    path = str(tmp_path / "extracted_priors.pkl")
    priors.save_priors(path, res, torch.zeros(3))
    with open(path, "rb") as f:
        p = pickle.load(f)
    xyz, feats, hits = read_priors_like_city_prior(p)
    m = res["points"].shape[0]
    assert m > 0 and xyz.shape == (m, 3) and feats.shape == (m, 64) and hits.shape == (m, 1)
    assert torch.isfinite(res["colors"]).all() and float(res["colors"].max()) <= 1.0
