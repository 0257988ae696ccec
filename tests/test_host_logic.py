"""Host-side logic of the product that needs no GPU: byte accounting, slice planning, fused-path eligibility, buffer
carving.  (The kernels themselves are only ever reached through CUDA tensors — tests/test_abi.py::test_no_cpu_fallback.)"""
import torch

from presight_b200 import fused, ops, synthetic


def test_algorithmic_bytes_match_survey():
    """SURVEY §8d: hash grid bytes per point and whole-step bytes per ray of the named configurations."""
    assert synthetic.hash_bytes_fwd(16, 2) == 1164 and synthetic.hash_bytes_bwd(16, 2) == 2188
    assert synthetic.hash_bytes_fwd(10, 4) == 1452 and synthetic.hash_bytes_bwd(10, 4) == 2732
    assert synthetic.hash_bytes_fwd(8, 1) == 300 and synthetic.hash_bytes_bwd(8, 1) == 556
    assert synthetic.hash_bytes_fwd(5, 2) == 372 and synthetic.hash_bytes_bwd(5, 2) == 692
    c1, c2 = synthetic.config_c1(), synthetic.config_c2()
    assert synthetic.step_bytes_per_ray(c1, True) == 535424 and synthetic.step_bytes_per_ray(c2, True) == 378880
    # non-update steps: proposal nets run without a backward
    assert synthetic.step_bytes_per_ray(c1, False) == 291840 and synthetic.step_bytes_per_ray(c2, False) == 272128


def test_chunk_bounds_are_the_whole_batch():
    for n, s in [(65536, 64), (65536, 128), (21846, 64), (100, 64), (40000, 64), (32768 + 5, 96)]:
        assert fused._chunk_bounds(n, s) == [(0, n)]            # the final level is never sliced


def test_fused_kernel_eligibility():
    """The tcgen05 level kernels implement exactly the reference field / proposal architectures (DESIGN §7)."""
    g_main = fused.GridMeta(tuple(float(i) for i in range(16)), 22, 2)
    base, sem, rgb = fused.MlpMeta((32, 64, 80), ops.ACT_NONE), fused.MlpMeta((64, 64, 64, 64), ops.ACT_NONE), \
        fused.MlpMeta((47, 64, 64, 3), ops.ACT_SIGMOID)
    ok = dict(grid=g_main, base=base, sem=sem, rgb=rgb, geo_dim=15, prec=ops.PREC_BF16, S=64, A=16)
    assert fused.tc5_field_supported(**ok)
    assert not fused.tc5_field_supported(**{**ok, "S": 48})                      # C1's final level
    assert not fused.tc5_field_supported(**{**ok, "prec": ops.PREC_TF32X3})      # fp32 class -> stand-alone kernels
    assert not fused.tc5_field_supported(**{**ok, "sem": None})
    assert not fused.tc5_field_supported(**{**ok, "A": 32, "rgb": fused.MlpMeta((63, 64, 64, 3), ops.ACT_SIGMOID)})
    g_prop = fused.GridMeta(tuple(float(i) for i in range(8)), 20, 1)
    net = fused.MlpMeta((8, 64, 1), ops.ACT_NONE)
    assert fused.tc5_prop_supported(g_prop, net, ops.PREC_BF16, 128) and fused.tc5_prop_supported(g_prop, net, ops.PREC_BF16, 96)
    assert not fused.tc5_prop_supported(g_prop, net, ops.PREC_BF16, 256)          # C1's first level
    assert not fused.tc5_prop_supported(g_prop, fused.MlpMeta((8, 32, 1), ops.ACT_NONE), ops.PREC_BF16, 64)
    g5 = fused.GridMeta(tuple(float(i) for i in range(5)), 17, 2)                 # C1 proposal grids: L5 F2, hidden 16
    assert fused.tc5_prop_supported(g5, fused.MlpMeta((10, 16, 1), ops.ACT_NONE), ops.PREC_BF16, 96)


def test_zeros_like_many_carves_aligned_views():
    ts = [torch.ones(3, 5), torch.ones(7), torch.ones(64, 64), torch.ones(1)]
    zs = ops.zeros_like_many(ts)
    assert [z.shape for z in zs] == [t.shape for t in ts]
    assert all(float(z.abs().sum()) == 0.0 and z.is_contiguous() for z in zs)
    assert all(z.data_ptr() % 16 == 0 for z in zs)
    base = zs[0].untyped_storage().data_ptr()
    assert all(z.untyped_storage().data_ptr() == base for z in zs)               # one allocation, one fill
    zs[1].add_(1.0)
    assert float(zs[0].sum()) == 0.0 and float(zs[2].sum()) == 0.0               # views do not overlap


def test_line_of_sight_schedules():
    from presight_b200.model import NerfactoNuscMSModel
    m = NerfactoNuscMSModel.__new__(NerfactoNuscMSModel)          # schedules only read the config
    m.config = synthetic.config_c2()
    assert m.get_line_of_sight_sigma(0) == 5.0 and m.get_line_of_sight_sigma(30000) == 2.0
    assert abs(m.get_line_of_sight_sigma(15500) - 3.5) < 1e-12
    assert m.get_line_of_sight_mult(1000) == 0.0 and m.get_line_of_sight_mult(1001) == 0.1
    assert m.get_line_of_sight_mult(12000) == 0.025
