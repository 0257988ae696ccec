"""CPU checks of the geometry metrics: the depth-metrics core (presight_b200/csrc/depth_metrics_core.h, the code the CUDA
kernels run) compiled for the host against the numpy fp64 oracle; the nearest-neighbour oracle (cKDTree) against brute
force; the grid's cell keys and its 2^21-cells-per-axis check."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from oracle import geometry_oracle as GO

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def host_lib(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("depth_metrics") / "libdepth_metrics_host.so")
    src = os.path.join(HERE, "native", "depth_metrics_host.cpp")
    subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-ffp-contract=off", src, "-o", out], check=True)
    lib = ctypes.CDLL(out)
    lib.depth_metrics_host.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_void_p, ctypes.c_float,
                                       ctypes.c_float, ctypes.c_float, ctypes.c_void_p]
    return lib


def run(lib, preds, target, scale, min_m=1.0, max_m=75.0):
    pred = np.ascontiguousarray(np.stack([np.asarray(p, np.float32).reshape(-1) for p in preds]))
    tgt = np.ascontiguousarray(np.asarray(target, np.float32).reshape(-1))
    out = np.zeros((len(preds), 8))
    rc = lib.depth_metrics_host(pred.ctypes.data, len(preds), tgt.size, tgt.ctypes.data, scale, min_m, max_m,
                                out.ctypes.data)
    return rc, out


def depth_case(H, W, M, seed, scale=0.0123):
    """M predicted maps (scene units) and a LiDAR-like target (metres, 0 where there is no return) with every edge case:
    targets at exactly min_m / max_m, predictions below, above and far outside the clamp."""
    rng = np.random.default_rng(seed)
    t = rng.uniform(0.2, 90.0, (H, W)).astype(np.float32)
    t[rng.random((H, W)) < 0.3] = 0.0
    t.flat[::17] = 1.0
    t.flat[5::19] = 75.0
    preds = []
    for m in range(M):
        p_m = t * np.exp(rng.normal(0.0, 0.1 + 0.1 * m, (H, W)))
        p_m.flat[3::11] = rng.uniform(-5.0, 0.9, p_m.flat[3::11].shape)     # below the clamp, negative too
        p_m.flat[7::13] = rng.uniform(76.0, 1e4, p_m.flat[7::13].shape)     # above it
        preds.append((p_m * scale).astype(np.float32))
    return preds, t


def assert_depth_close(got, want, rel=1e-12):
    assert got.shape == want.shape
    np.testing.assert_array_equal(got[:, 7], want[:, 7])
    n = want[:, 7]
    for m in range(len(want)):
        if n[m] == 0:
            assert np.isnan(got[m, :7]).all() and np.isnan(want[m, :7]).all()
            continue
        # the delta terms are counts: exact
        np.testing.assert_array_equal(np.round(got[m, 4:7] * n[m]), np.round(want[m, 4:7] * n[m]))
        np.testing.assert_allclose(got[m, :7], want[m, :7], rtol=rel, atol=0)


@pytest.mark.parametrize("M", [1, 2, 4])
@pytest.mark.parametrize("H,W", [(31, 31), (90, 160)])
def test_depth_core_matches_oracle(host_lib, H, W, M):
    preds, t = depth_case(H, W, M, seed=H + M)
    rc, got = run(host_lib, preds, t, 0.0123)
    assert rc == 0
    want = GO.depth_metrics(preds, t, 0.0123)
    assert_depth_close(got, want)
    assert 0 < want[0, 7] < H * W


def test_targets_at_the_bounds_and_zero_are_not_valid(host_lib):
    t = np.array([0.0, 1.0, 75.0, 1.0000001, 74.99999, 30.0], np.float32)
    p = np.array([5.0, 5.0, 5.0, 5.0, 5.0, 5.0], np.float32)
    _, got = run(host_lib, [p], t, 1.0)
    want = GO.depth_metrics([p], t, 1.0)
    assert got[0, 7] == want[0, 7] == 3
    assert_depth_close(got, want)


def test_predictions_are_clamped(host_lib):
    t = np.array([10.0, 10.0, 2.0, 70.0], np.float32)
    p = np.array([-3.0, 1e6, 0.5, np.float32(80.0)], np.float32)
    _, got = run(host_lib, [p], t, 1.0)
    clamped = np.array([1.0, 75.0, 1.0, 75.0])
    d = clamped - t
    assert got[0, 0] == pytest.approx(np.mean(np.abs(d) / t), rel=1e-15)
    assert got[0, 2] == pytest.approx(np.sqrt(np.mean(d * d)), rel=1e-15)
    assert_depth_close(got, GO.depth_metrics([p], t, 1.0))


def test_no_valid_pixel_gives_nan(host_lib):
    t = np.array([0.0, 0.5, 1.0, 75.0, 80.0], np.float32)
    preds = [np.ones(5, np.float32), 3 * np.ones(5, np.float32)]
    rc, got = run(host_lib, preds, t, 1.0)
    assert rc == 0
    assert np.isnan(got[:, :7]).all() and (got[:, 7] == 0).all()
    assert_depth_close(got, GO.depth_metrics(preds, t, 1.0))


def test_perfect_prediction_and_map_count(host_lib):
    preds, t = depth_case(20, 30, 1, seed=3, scale=1.0)
    exact = np.clip(t, 1.0, 75.0)
    _, got = run(host_lib, [exact], t, 1.0)
    assert (got[0, :4] == 0).all() and (got[0, 4:7] == 1).all()
    assert run(host_lib, preds * 5, t, 1.0)[0] == 1


# ---- nearest neighbours ---------------------------------------------------------------------------------------------
def nn_cases():
    rng = np.random.default_rng(11)
    r = 0.5
    cases = {"random": (rng.uniform(-3, 3, (300, 3)), rng.uniform(-3, 3, (400, 3)), 0.7)}
    ref = rng.uniform(-2, 2, (200, 3))
    cases["duplicates"] = (np.concatenate([ref, ref[:50]]), np.concatenate([ref[::3], ref[::3], ref[:5] + 0.01]), 0.3)
    cases["negative"] = (rng.uniform(-1000.5, -999.5, (150, 3)), rng.uniform(-1000.5, -999.5, (170, 3)), 0.25)
    g = np.arange(6) * r                                           # points exactly one cell (and r) apart
    lattice = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3)
    cases["one_cell_apart"] = (lattice + np.array([0.0, 0.0, r / 2]), lattice, r)
    cases["one_point"] = (rng.uniform(-1, 1, (60, 3)), np.array([[0.1, -0.2, 0.3]]), 1.0)
    return cases


@pytest.mark.parametrize("name", list(nn_cases()))
def test_nn_oracle_matches_brute_force(name):
    q, p, r = nn_cases()[name]
    q, p = q.astype(np.float32), p.astype(np.float32)
    want = GO.nn_distances_brute(q, p, r)
    got = GO.nn_distances(q, p, r)
    np.testing.assert_allclose(got, want, rtol=1e-15, atol=0)
    assert (got <= r).all()
    for tau in (r / 4, r / 2, r):
        assert int((got < tau).sum()) == int((want < tau).sum())


def test_nn_exactly_r_apart_is_clamped():
    q, p, r = nn_cases()["one_cell_apart"]
    d = GO.nn_distances(q.astype(np.float32), p.astype(np.float32), r)
    np.testing.assert_array_equal(d, np.full(len(q), r / 2))
    far = GO.nn_distances(np.array([[0.0, 0.0, 1.0]], np.float32), np.array([[0.0, 0.0, 0.0]], np.float32), 1.0)
    assert far[0] == 1.0                                           # distance == r is not < r


def test_prior_metrics_oracle_definitions():
    q, p, r = nn_cases()["random"]
    m = GO.prior_geometry_metrics(q.astype(np.float32), p.astype(np.float32), r, (0.1, 0.35, 0.7))
    assert m["accuracy"] == pytest.approx(GO.nn_distances_brute(q, p, r).mean(), rel=1e-14)
    assert m["completeness"] == pytest.approx(GO.nn_distances_brute(p, q, r).mean(), rel=1e-14)
    P, R = m["precision"], m["recall"]
    np.testing.assert_allclose(m["fscore"], 2 * P * R / (P + R))
    assert (np.diff(P) >= 0).all() and (np.diff(R) >= 0).all()


# ---- cell keys ------------------------------------------------------------------------------------------------------
def test_cell_keys_pack_21_bits_per_axis():
    rng = np.random.default_rng(2)
    pts = rng.uniform(-50, 30, (1000, 3)).astype(np.float32)
    r = 0.4
    origin = pts.min(axis=0)
    keys = GO.cell_keys(pts, origin, r)
    c = GO.cell_coords(pts, origin, r)
    assert (c >= 0).all() and (c < (1 << 21)).all() and (c.min(axis=0) == 0).all()
    np.testing.assert_array_equal(GO.unpack_cell_keys(keys), c)
    order = np.argsort(keys, kind="stable")                        # key order is (x, y, z) lexicographic
    np.testing.assert_array_equal(np.lexsort((c[order, 2], c[order, 1], c[order, 0])), np.arange(len(pts)))
    top = np.array([[(1 << 21) - 1] * 3])
    np.testing.assert_array_equal(GO.unpack_cell_keys(GO.cell_keys(top.astype(np.float32), [0, 0, 0], 1.0)), top)


@pytest.fixture(scope="module")
def lib():
    from presight_b200 import _lib, build
    if not os.path.exists(_lib.LIB_PATH):
        build.build(verbose=False)
    return _lib.load()


def cells_per_axis_native(lib, pts, r):
    pts = np.asarray(pts, np.float32)
    b = (ctypes.c_float * 6)(*pts.min(axis=0).tolist(), *pts.max(axis=0).tolist())
    cells = (ctypes.c_int64 * 3)()
    rc = lib.ps_nn_grid_cells_per_axis(b, r, cells)
    return rc, list(cells)


def test_extent_check(lib):
    r = 0.5
    ok = np.array([[0, -3, 7], [((1 << 21) - 1) * r, -3 + 10 * r, 7]], np.float32)   # exactly 2^21 cells on x
    rc, cells = cells_per_axis_native(lib, ok, r)
    assert rc == 0 and cells == [1 << 21, 11, 1]
    np.testing.assert_array_equal(GO.cells_per_axis(ok, r), cells)
    bad = ok.copy()
    bad[1, 0] = (1 << 21) * r                                                    # one cell more
    rc, _ = cells_per_axis_native(lib, bad, r)
    assert rc == 1 and b"2^21" in lib.ps_last_error()
    with pytest.raises(ValueError):
        GO.cells_per_axis(bad, r)
    rc, _ = cells_per_axis_native(lib, np.array([[0, 0, 0], [1, 1, 1e6]], np.float32), 0.4)
    assert rc == 1 and b"axis 2" in lib.ps_last_error()
    for bad_r in (0.0, -1.0, float("inf"), float("nan")):
        assert cells_per_axis_native(lib, ok, bad_r)[0] == 1
    # the ABI refuses the keys of an over-wide set before touching any device pointer
    b = (ctypes.c_float * 6)(0, 0, 0, (1 << 21) * r, 1, 1)
    assert lib.ps_nn_grid_keys(1, 2, b, r, 1, None) == 1
