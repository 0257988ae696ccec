"""CPU checks of prior extraction: the per-ray surface-hit core (presight_b200/csrc/hits_core.h, the code the CUDA kernel
runs per thread) compiled for the host, the eligibility rule of the fused density level, and the byte model of the
depth pass."""
import ctypes
import os
import subprocess
from fractions import Fraction

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def host_lib(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("hits") / "libhits_host.so")
    src = os.path.join(HERE, "native", "hits_host.cpp")
    subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-ffp-contract=off", src, "-o", out], check=True)
    lib = ctypes.CDLL(out)
    lib.surface_hits_host.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_float,
                                      ctypes.c_float, ctypes.c_float, ctypes.c_float, ctypes.c_void_p, ctypes.c_void_p,
                                      ctypes.c_void_p]
    return lib


def run(lib, o, d, t, scale, max_range=np.nan, z_min=np.nan, z_max=np.nan):
    o, d, t = (np.ascontiguousarray(a, dtype=np.float32) for a in (o, d, t))
    n = t.shape[0]
    ps, pm = np.zeros((n, 3), np.float32), np.zeros((n, 3), np.float32)
    keep = np.zeros(n, np.uint8)
    assert lib.surface_hits_host(o.ctypes.data, d.ctypes.data, t.ctypes.data, n, scale, max_range, z_min, z_max,
                                 ps.ctypes.data, pm.ctypes.data, keep.ctypes.data) == 0
    return ps, pm, keep.astype(bool)


def fma_f32(a, b, c):
    """Correctly rounded float32 a * b + c (round to nearest, ties to even), from exact rational arithmetic."""
    exact = Fraction(float(a)) * Fraction(float(b)) + Fraction(float(c))
    g = np.float32(float(exact))
    cands = [np.nextafter(g, np.float32(-np.inf)), g, np.nextafter(g, np.float32(np.inf))]
    errs = [abs(Fraction(float(x)) - exact) for x in cands]
    best = min(errs)
    ties = [x for x, e in zip(cands, errs) if e == best]
    return ties[0] if len(ties) == 1 else [x for x in ties if (x.view(np.int32) & 1) == 0][0]


def test_hit_points_are_one_fma_and_one_division(host_lib):
    rng = np.random.default_rng(0)
    n = 3000
    o = (rng.standard_normal((n, 3)) * 5).astype(np.float32)
    d = rng.standard_normal((n, 3)).astype(np.float32)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    t = (rng.random(n) * 20).astype(np.float32)
    scale = np.float32(0.05)
    ps, pm, keep = run(host_lib, o, d, t, scale)
    want = np.array([[fma_f32(d[i, k], t[i], o[i, k]) for k in range(3)] for i in range(n)], dtype=np.float32)
    assert np.array_equal(ps.view(np.int32), want.view(np.int32))
    # one rounding, not two: the unfused form differs somewhere
    assert not np.array_equal(ps, (d * t[:, None]).astype(np.float32) + o)
    assert np.array_equal(pm.view(np.int32), (ps / scale).astype(np.float32).view(np.int32))
    assert keep.all()                                         # no bound given


def test_selector_boundaries_and_non_finite_bounds(host_lib):
    scale = np.float32(0.05)
    # straight up rays from z = 0: points_m.z = depth / scale, range_m = depth / scale
    z_m = np.array([1.0, 2.0, 3.0, 4.0], np.float32)
    t = (z_m * scale).astype(np.float32)
    o = np.zeros((4, 3), np.float32)
    d = np.tile(np.array([0, 0, 1], np.float32), (4, 1))
    _, pm, _ = run(host_lib, o, d, t, scale)
    r = (t / scale).astype(np.float32)                        # the range the core compares
    z = pm[:, 2]
    # range: <= is inclusive
    _, _, k = run(host_lib, o, d, t, scale, max_range=r[1])
    assert k.tolist() == [True, True, False, False]
    _, _, k = run(host_lib, o, d, t, scale, max_range=np.nextafter(r[1], np.float32(0)))
    assert k.tolist() == [True, False, False, False]
    # height window: both ends inclusive
    _, _, k = run(host_lib, o, d, t, scale, z_min=z[1], z_max=z[2])
    assert k.tolist() == [False, True, True, False]
    _, _, k = run(host_lib, o, d, t, scale, z_min=np.nextafter(z[1], np.float32(np.inf)), z_max=z[2])
    assert k.tolist() == [False, False, True, False]
    # a bound that is not finite is not applied
    for inf_like in (np.inf, -np.inf, np.nan):
        _, _, k = run(host_lib, o, d, t, scale, max_range=inf_like, z_min=inf_like, z_max=inf_like)
        assert k.all(), inf_like
    _, _, k = run(host_lib, o, d, t, scale, max_range=np.nan, z_min=-np.inf, z_max=z[0])
    assert k.tolist() == [True, False, False, False]


def test_tc5_density_supported():
    from presight_b200 import fused, ops
    g = fused.GridMeta
    c2 = g(tuple(range(16)), 22, 2)          # L16 F2: K0 = 32
    shipped = g(tuple(range(10)), 20, 4)     # L10 F4: K0 = 48
    small = g(tuple(range(6)), 19, 2)        # L6 F2:  K0 = 16
    for grid in (c2, shipped, small, g(tuple(range(12)), 19, 4), g(tuple(range(48)), 19, 1)):
        for S in (32, 64, 96, 128):
            assert fused.tc5_density_supported(grid, 64, ops.PREC_BF16, S)
    assert not fused.tc5_density_supported(c2, 64, ops.PREC_TF32X3, 64)        # fp32 class keeps the old path
    assert not fused.tc5_density_supported(c2, 64, ops.PREC_BF16, 48)          # C1's final level
    assert not fused.tc5_density_supported(c2, 32, ops.PREC_BF16, 64)          # hidden width
    assert not fused.tc5_density_supported(g(tuple(range(13)), 19, 4), 64, ops.PREC_BF16, 64)   # L*F = 52 > 48
    assert not fused.tc5_density_supported(g(tuple(range(8)), 19, 8), 64, ops.PREC_BF16, 64)    # F = 8


def test_depth_pass_bytes_per_ray():
    from presight_b200 import synthetic
    assert synthetic.depth_pass_bytes_per_ray(synthetic.config_c2()) == 132096
    assert synthetic.depth_pass_bytes_per_ray(synthetic.config_presight()) == 150528
