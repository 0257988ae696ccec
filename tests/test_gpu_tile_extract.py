"""A whole tile's priors in bounded device memory: ps_hits_append against nonzero + gather, TileVoxelizer against
postprocess_priors and the reference fixture, PriorExtractor on small store blocks against the public pieces composed by
hand, and TileVoxelizer at 2^28 points with exactly known voxel means and a bound on its device memory."""
import types

import numpy as np
import pytest
import torch

from helpers import Fixture
from test_gpu_extract import c2_model, presight_model, synth_bundle

pytestmark = pytest.mark.gpu
DEV = "cuda"


def random_chunk(n, seed, colors=True, dens_scale=1.0):
    g = torch.Generator(device=DEV).manual_seed(seed)
    ps = torch.randn(n, 3, device=DEV, generator=g) * 20.0
    pm = ps / torch.full((1, 3), 0.05, device=DEV)
    keep = torch.rand(n, device=DEV, generator=g) < 0.6
    dens = torch.rand(n, device=DEV, generator=g) * 2.0 * dens_scale
    col = torch.rand(n, 3, device=DEV, generator=g) if colors else None
    return ps, pm, keep, dens, col


def torch_tail(ps, pm, keep, dens, col):
    idx = torch.nonzero(keep & (dens > 1)).view(-1)
    c = torch.zeros(idx.numel(), 3, device=DEV) if col is None else col[idx]
    return ps[idx], c, pm[idx]


class Store:
    def __init__(self, capacity, n_max):
        import ctypes as C
        from presight_b200._lib import load
        self.cap = capacity
        self.pts = torch.full((capacity, 3), float("nan"), device=DEV)
        self.cols = torch.full((capacity, 3), float("nan"), device=DEV)
        self.cursor = torch.zeros(1, device=DEV, dtype=torch.int64)
        self.min = torch.full((3,), float("inf"), device=DEV)
        self.status = torch.zeros(1, device=DEV, dtype=torch.int32)
        nbytes = C.c_int64()
        assert load().ps_hits_append_workspace(n_max, C.byref(nbytes)) == 0
        self.ws = torch.empty(nbytes.value, device=DEV, dtype=torch.uint8)

    def append(self, ps, pm, keep, dens, col):
        from presight_b200._lib import call, ptr, stream
        call("ps_hits_append", ptr(ps), ptr(pm), ptr(keep), ptr(dens), ptr(col), ps.shape[0], ptr(self.pts),
             ptr(self.cols), self.cap, ptr(self.cursor), ptr(self.min), ptr(self.status), ptr(self.ws), stream())


@pytest.mark.parametrize("colors", [True, False])
def test_hits_append_matches_nonzero_gather(colors):
    from presight_b200.priors import PriorVoxelizer
    sizes = [5000, 1, 3000, 300000, 0, 2047, 777]
    st = Store(1 << 20, max(sizes))
    want_p, want_c, want_m = [], [], []
    for k, n in enumerate(sizes):
        chunk = random_chunk(n, seed=k, colors=colors)
        st.append(*chunk)
        p, c, m = torch_tail(*chunk)
        want_p.append(p), want_c.append(c), want_m.append(m)
        assert int(st.cursor) == sum(x.shape[0] for x in want_p)
    wp, wc, wm = torch.cat(want_p), torch.cat(want_c), torch.cat(want_m)
    n = wp.shape[0]
    assert n > 50000
    assert torch.equal(st.pts[:n], wp) and torch.equal(st.cols[:n], wc)
    assert torch.equal(st.min, PriorVoxelizer.min_bound(wm))
    assert bool(st.pts[n:].isnan().all()) and int(st.status) == 0


def test_hits_append_keeps_nothing_and_refuses_overflow():
    st = Store(4000, 20000)
    st.append(*random_chunk(10000, seed=3, dens_scale=0.5))          # every density <= 1
    assert int(st.cursor) == 0 and bool(torch.isinf(st.min).all()) and int(st.status) == 0
    first = random_chunk(3000, seed=4)
    st.append(*first)
    c0 = int(st.cursor)
    assert 0 < c0 < 4000
    snap_p, snap_min = st.pts.clone(), st.min.clone()
    st.append(*random_chunk(20000, seed=5))                            # ~6000 more rows: does not fit
    assert int(st.status) & 1
    assert int(st.cursor) == c0 and torch.equal(st.min, snap_min)
    assert torch.equal(st.pts[:c0], snap_p[:c0]) and bool(st.pts[c0:].isnan().all())


@pytest.mark.parametrize("colors", [True, False])
def test_extractor_store_blocks_across_a_boundary(colors):
    """PriorExtractor's host side over ps_hits_append with blocks of 5000 hits: the filled views of the blocks are the
    kept rows in ray order, and the running minimum is the one of all of them."""
    from presight_b200.extract import PriorExtractor
    from presight_b200.priors import PriorVoxelizer
    ex = PriorExtractor(types.SimpleNamespace(training=False), 0.05, chunk_rays=4096, block_hits=5000)
    want_p, want_c, want_m = [], [], []
    for k in range(9):
        ps, pm, keep, dens, col = random_chunk(4096 - 100 * k, seed=10 + k, colors=colors)
        if k == 4:
            dens = dens * 0.25                                          # a chunk that keeps nothing
        ex._append(ps, pm, keep.to(torch.uint8), dens, col)
        p, c, m = torch_tail(ps, pm, keep, dens, col)
        want_p.append(p), want_c.append(c), want_m.append(m)
    assert len(ex._blocks) > 2 and all(k <= 5000 for k in ex._filled())
    assert ex.n_hits == sum(p.shape[0] for p in want_p)
    assert torch.equal(torch.cat(ex._points), torch.cat(want_p))
    cols = torch.cat([c[:k] for (_, c), k in zip(ex._blocks, ex._filled())])
    assert torch.equal(cols, torch.cat(want_c))
    assert torch.equal(ex._min, PriorVoxelizer.min_bound(torch.cat(want_m)))
    assert int(ex._status) == 0


def tile_voxelize(pts, feats, cols, mn, vs, q, slice_, capacity):
    from presight_b200.priors import TileVoxelizer
    vox = TileVoxelizer(mn, vs, feats.shape[1], capacity=capacity)
    for i in range(0, pts.shape[0], slice_):
        vox.insert(pts[i:i + slice_])
    vox.seal()
    for i in range(0, pts.shape[0], slice_):
        vox.accumulate(pts[i:i + slice_], feats[i:i + slice_], cols[i:i + slice_])
    return vox, vox.finalize(q)


def assert_same_priors(got, want):
    assert got["n_voxels"] == want["n_voxels"]
    assert float(got["hit_thr"]) == float(want["hit_thr"])
    assert torch.equal(got["hits"], want["hits"])
    assert torch.equal(got["features"], want["features"])
    np.testing.assert_allclose(got["points"].cpu().numpy(), want["points"].cpu().numpy(), rtol=1e-6, atol=1e-6)
    np.testing.assert_allclose(got["colors"].cpu().numpy(), want["colors"].cpu().numpy(), rtol=2e-6, atol=1e-7)


@pytest.mark.parametrize("case", ["a", "b", "c"])
def test_tile_voxelizer_matches_reference_fixture(case):
    from presight_b200 import priors
    fx = Fixture("priors.npz")
    g = lambda k: fx.np(f"{case}/{k}")
    P, Fh, C, D = (torch.from_numpy(np.ascontiguousarray(g(k))).to(DEV)
                   for k in ("in_points", "in_features", "in_colors", "in_densities"))
    vs, q = float(g("voxel_size")), float(g("hit_thr_ratio"))
    sel = D > 1
    mn = priors.PriorVoxelizer.min_bound(P, D)
    _, out = tile_voxelize(P[sel].float(), Fh[sel].half(), C[sel].float(), mn, vs, q, 1 << 20, 1 << 16)
    assert out["n_voxels"] == int(g("n_voxels"))
    assert float(out["hit_thr"]) == float(g("hit_thr"))
    np.testing.assert_array_equal(out["hits"].cpu().numpy(), g("hits"))
    np.testing.assert_array_equal(out["features"].cpu().numpy(), g("features"))
    np.testing.assert_allclose(out["points"].cpu().numpy(), g("points"), rtol=1e-6, atol=1e-6)
    np.testing.assert_allclose(out["colors"].cpu().numpy(), g("colors"), rtol=2e-6, atol=1e-7)
    assert_same_priors(out, priors.postprocess_priors(P, Fh, C, D, vs, q))


def test_tile_voxelizer_grows_its_table():
    """Random points, a 4-slot initial table and slices of 257 points: the table is rehashed many times."""
    from presight_b200 import priors
    g = torch.Generator(device=DEV).manual_seed(7)
    n = 200000
    pts = torch.rand(n, 3, device=DEV, generator=g) * torch.tensor([60.0, 30.0, 6.0], device=DEV) - 10.0
    feats = torch.rand(n, 64, device=DEV, generator=g).half()
    cols = torch.rand(n, 3, device=DEV, generator=g)
    mn = priors.PriorVoxelizer.min_bound(pts)
    vox, out = tile_voxelize(pts, feats, cols, mn, 0.4, 0.2, 257, 4)
    assert vox.capacity >= 2 * out["n_voxels"] and out["n_voxels"] > 50000
    assert_same_priors(out, priors.postprocess_priors(pts, feats, cols, None, 0.4, 0.2))


@pytest.mark.parametrize("shape", ["c2", "presight16"])
def test_extractor_blocks_and_growth_match_hand_composition(shape):
    from presight_b200 import priors
    from presight_b200.cameras.rays import RayBundle
    from presight_b200.extract import PriorExtractor, surface_hits
    model, _ = c2_model() if shape == "c2" else presight_model()
    n = 20000
    rb = synth_bundle(n, seed=13)
    colors = torch.rand(n, 3, generator=torch.Generator().manual_seed(2)).to(DEV)
    kw = dict(max_range_m=60.0, z_range_m=(-3.0, 12.0))
    ex = PriorExtractor(model, 0.05, chunk_rays=2500, block_hits=2500, insert_slice=64, **kw)
    ex.add(rb, colors)
    got = ex.finalize()
    with torch.no_grad():
        depth = model.get_surface_hits(RayBundle(origins=rb.origins, directions=rb.directions))["depth"]
        ps, pm, keep = surface_hits(rb.origins, rb.directions, depth, 0.05, **kw)
        dens, feats = model.query_priors(ps)
        k = keep & (dens > 1)
        ref = priors.postprocess_priors(pm[k], feats[k], colors[k], None)
    # blocks of one chunk: two chunks with kept hits never share a block
    chunks_with_hits = len(set((torch.nonzero(k).view(-1) // 2500).tolist()))
    assert len(ex._blocks) >= chunks_with_hits
    assert shape == "c2" or chunks_with_hits > 1
    assert torch.equal(torch.cat(ex._points) / torch.full((1, 3), 0.05, device=DEV), pm[k])
    assert ex.n_hits == int(k.sum())
    assert_same_priors(got, ref)


def test_tile_voxelizer_at_scale():
    """2^28 points into 2^19 voxels of a 128 x 128 x 32 lattice.  Point i lies in voxel floor(k^2 / 2^37), k = i * A mod
    2^28 (a bijection, so every voxel is hit, from ~256 to ~370 000 times); its features and colour are functions of
    its voxel only, so the means are known exactly.  The voxelizer's device memory beyond the resident points is
    bounded by its table, its rows and one slice -- the points-sized table of PriorVoxelizer would need 397 GB."""
    from presight_b200.priors import TileVoxelizer
    H, V, C, vs = 1 << 28, 1 << 19, 64, 0.4
    P_ins, P_acc = 1 << 24, 1 << 21
    A = 0x9E3779B1

    def voxel_of(i0, n):
        k = (torch.arange(i0, i0 + n, device=DEV, dtype=torch.int64) * A) & (H - 1)
        return (k * k) >> 37

    def cell(vid):
        return torch.stack([vid & 127, (vid >> 7) & 127, vid >> 14], 1)

    def feat_of(vid):
        c = torch.arange(C, device=DEV, dtype=torch.int32)
        return (((vid.int()[:, None] * 13 + c * 7) % 2048).float() / 64.0).half()

    def col_of(vid):
        a = torch.arange(3, device=DEV, dtype=torch.int64)
        return ((vid[:, None] + a * 97) % 256).float() / 256.0

    torch.cuda.empty_cache()
    g = torch.Generator(device=DEV).manual_seed(0)
    pts = torch.empty(H, 3, device=DEV)
    counts = torch.zeros(V, device=DEV, dtype=torch.int64)
    for i0 in range(0, H, P_ins):
        vid = voxel_of(i0, P_ins)
        jit = torch.rand(P_ins, 3, device=DEV, generator=g, dtype=torch.float64) * 0.8 + 0.1
        pts[i0:i0 + P_ins] = (-1.2 + vs * (cell(vid).double() + jit)).float()     # lattice anchor for min_point = 0
        counts += torch.bincount(vid, minlength=V)
        del vid, jit
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()

    vox = TileVoxelizer(torch.zeros(3, device=DEV), vs, C)
    for i0 in range(0, H, P_ins):
        vox.insert(pts[i0:i0 + P_ins])
    vox.seal()
    for i0 in range(0, H, P_acc):
        vid = voxel_of(i0, P_acc)
        vox.accumulate(pts[i0:i0 + P_acc], feat_of(vid), col_of(vid))
        del vid
    assert int(vox.counts.long().sum()) == H
    keys_all = cell(torch.arange(V, device=DEV))
    keys_all = (keys_all[:, 0] << 42) | (keys_all[:, 1] << 21) | keys_all[:, 2]
    order = torch.argsort(keys_all)
    assert torch.equal(vox.row_keys, keys_all[order])
    assert torch.equal(vox.counts.long(), counts[order])
    torch.cuda.synchronize()
    before_finalize = torch.cuda.max_memory_allocated()
    out = vox.finalize(0.2)
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base

    exp_hits = counts[order]
    thr = float(np.quantile(exp_hits.cpu().numpy(), 0.2))
    assert out["n_voxels"] == V and float(out["hit_thr"]) == thr
    kept = exp_hits.double() > thr
    vid_kept = torch.arange(V, device=DEV)[order][kept]
    assert torch.equal(out["hits"], exp_hits[kept])
    assert torch.equal(out["features"], feat_of(vid_kept))
    assert torch.equal(out["colors"], col_of(vid_kept))
    lo = (-1.2 + vs * cell(vid_kept).double())
    com = out["points"].double()
    assert bool(((com >= lo) & (com <= lo + vs)).all())
    # table slots (8 B key + 4 B row, <= 4 (V + P) slots after power-of-two rounding, the old table beside the new one
    # while rehashing) + 740 B per row (accumulators and outputs) twice over for the kept copies + one slice's
    # generated features and colours with their int32 / fp32 temporaries
    slice_bytes = P_acc * C * 16
    bound = 16 * 4 * (V + P_ins) + 2 * 740 * V + slice_bytes
    assert peak <= bound, (peak, bound, before_finalize - base)
