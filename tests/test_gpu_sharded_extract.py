"""One tile's extraction over several GPUs, the single-GPU parts: the owner partition of stored hits (ps_voxel_partition)
against a torch restatement of its key and owner hash, the hit quantile from summed histograms against ps_hits_quantile,
and ShardedPriorExtractor without a process group against PriorExtractor."""
import numpy as np
import pytest
import torch

from test_gpu_extract import c2_model, presight_model, synth_bundle
from test_gpu_tile_extract import assert_same_priors

pytestmark = pytest.mark.gpu
DEV = "cuda"
SCALE, VS = 0.05, 0.4


def _shr(x, s):                                   # logical right shift of int64 bit patterns
    return (x >> s) & ((1 << (64 - s)) - 1)


def _i64(c):                                      # a uint64 constant as the int64 with the same bits
    return c - (1 << 64) if c >= 1 << 63 else c


def owner_ref(keys, world):
    """The documented owner: (splitmix64(key) >> 32) % world, in int64 arithmetic (products wrap mod 2^64)."""
    z = keys ^ _shr(keys, 30)
    z = z * _i64(0xbf58476d1ce4e5b9)
    z = z ^ _shr(z, 27)
    z = z * _i64(0x94d049bb133111eb)
    z = z ^ _shr(z, 31)
    return _shr(z, 32) % world


def keys_ref(pts, anchor):
    """ps_voxel_insert's key of scene-unit points, restated: metres by IEEE division, open3d's floor in doubles."""
    pm = pts / torch.full((1, 3), SCALE, device=DEV)
    vmb = (anchor - 1.0).double() - VS * 0.5
    # divided by a tensor: torch turns a division by a Python scalar into a multiplication by its reciprocal
    idx = torch.floor((pm.double() - vmb) / torch.full((1, 3), VS, device=DEV, dtype=torch.float64)).long()
    ok = bool(((idx >= 0) & (idx < (1 << 21))).all())
    idx = idx & ((1 << 21) - 1)
    return (idx[:, 0] << 42) | (idx[:, 1] << 21) | idx[:, 2], ok


def partition(pts, cols, anchor, world):
    import ctypes as C
    from presight_b200._lib import call, check, load, ptr, stream
    n = pts.shape[0]
    nbytes = C.c_int64()
    check(load().ps_voxel_partition_workspace(n, world, C.byref(nbytes)), "ps_voxel_partition_workspace")
    ws = torch.full((nbytes.value,), 0xAB, device=DEV, dtype=torch.uint8)
    out_p = torch.full((n, 3), float("nan"), device=DEV)
    out_c = torch.full((n, 3), float("nan"), device=DEV)
    counts = torch.full((world,), -1, device=DEV, dtype=torch.int64)
    status = torch.zeros(1, device=DEV, dtype=torch.int32)
    call("ps_voxel_partition", ptr(pts), ptr(cols), n, SCALE, ptr(anchor), VS, world, ptr(out_p), ptr(out_c),
         ptr(counts), ptr(status), ptr(ws), stream())
    return out_p, out_c, counts, int(status)


def hits_input(kind):
    """-> scene-unit points, colours, lattice anchor (metres)."""
    g = torch.Generator(device=DEV).manual_seed({"random": 1, "one_voxel": 2, "boundaries": 3, "empty": 4}[kind])
    if kind == "random":
        pts = torch.randn(300000, 3, device=DEV, generator=g) * 20.0
    elif kind == "one_voxel":                     # every hit in one voxel: all lanes of every warp share an owner
        pts = (0.1 + torch.rand(100000, 3, device=DEV, generator=g) * 0.2) * SCALE     # voxel (3, 3, 3) of anchor 0
    elif kind == "boundaries":                    # hits within a few ulps of voxel faces, both sides
        k = torch.randint(1, 200, (50000, 3), device=DEV, generator=g).double()
        pm = (-1.2 + k * VS).float()
        for _ in range(2):
            step = torch.randint(-1, 2, pm.shape, device=DEV, generator=g).float()
            pm = torch.nextafter(pm, pm + step)
        pts = pm * SCALE
    else:
        pts = torch.empty(0, 3, device=DEV)
    pts = pts.contiguous()
    cols = torch.rand(pts.shape[0], 3, device=DEV, generator=g)
    pm = pts / torch.full((1, 3), SCALE, device=DEV)
    from presight_b200.priors import PriorVoxelizer
    anchor = PriorVoxelizer.min_bound(pm) if kind == "random" else torch.zeros(3, device=DEV)
    return pts, cols, anchor


@pytest.mark.parametrize("world", [1, 2, 3, 8])
@pytest.mark.parametrize("kind", ["random", "one_voxel", "boundaries", "empty"])
def test_partition_is_a_stable_sort_by_owner(kind, world):
    from presight_b200.priors import TileVoxelizer
    pts, cols, anchor = hits_input(kind)
    pm = pts / torch.full((1, 3), SCALE, device=DEV)
    out_p, out_c, counts, st = partition(pts, cols, anchor, world)
    assert st == 0
    keys, ok = keys_ref(pts, anchor)
    assert ok
    own = owner_ref(keys, world)
    perm = torch.cat([torch.nonzero(own == r).view(-1) for r in range(world)])
    assert torch.equal(counts, torch.bincount(own, minlength=world))
    assert torch.equal(out_p, pts[perm]) and torch.equal(out_c, cols[perm])   # once each, owner segments, input order
    if not pts.shape[0]:
        return
    bounds = [0] + torch.cumsum(counts, 0).tolist()
    seg_keys = [torch.unique(keys_ref(out_p[bounds[r]:bounds[r + 1]], anchor)[0]) for r in range(world)]
    for r in range(world):
        assert bool((owner_ref(seg_keys[r], world) == r).all())
    vox = TileVoxelizer(anchor, VS, 0)
    vox.insert(pm)
    vox.seal()
    union = torch.cat(seg_keys)
    assert torch.unique(union).numel() == union.numel()                      # the owners' voxel sets are disjoint
    assert torch.equal(torch.sort(union).values, vox.row_keys)
    if kind == "boundaries":
        assert vox.row_keys.numel() > 40000
    if kind == "one_voxel":
        assert vox.row_keys.numel() == 1 and int((counts > 0).sum()) == 1


def test_partition_flags_a_key_outside_21_bits():
    pts, cols, anchor = hits_input("random")
    pts = pts[:5000].clone()
    pts[1234] = torch.tensor([1.0e6 * SCALE, 0.0, 0.0], device=DEV)          # 10^6 m from the anchor: 2.5 M voxels
    out_p, _, counts, st = partition(pts, cols[:5000], anchor, 3)
    assert st & 2
    assert int(counts.sum()) == 5000 and not bool(out_p.isnan().any())


def hits_quantile(hits, q, bins):
    from presight_b200._lib import call, ptr, stream
    hist = torch.zeros(bins, device=DEV, dtype=torch.int32)
    thr = torch.zeros(1, device=DEV, dtype=torch.float64)
    st = torch.zeros(1, device=DEV, dtype=torch.int32)
    call("ps_hits_quantile", ptr(hits), hits.numel(), float(q), ptr(hist), bins, ptr(thr), ptr(st), stream())
    assert int(st) == 0
    return thr


@pytest.mark.parametrize("q", [0.0, 0.2, 0.5, 1.0])
@pytest.mark.parametrize("kind", ["random", "one_voxel", "all_equal"])
def test_summed_histogram_quantile_matches_hits_quantile(kind, q):
    from presight_b200._lib import call, ptr, stream
    g = torch.Generator(device=DEV).manual_seed(11)
    if kind == "random":
        hits = torch.randint(1, 700, (100003,), device=DEV, generator=g)
    elif kind == "one_voxel":
        hits = torch.tensor([7], device=DEV)
    else:
        hits = torch.full((4099,), 3, device=DEV, dtype=torch.int64)
    M, bins = hits.numel(), int(hits.max()) + 1
    want = hits_quantile(hits, q, bins)
    assert float(want) == float(np.quantile(hits.cpu().numpy(), q))
    k = 5                                         # k random parts, some of them empty when M < k
    perm = torch.randperm(M, device=DEV, generator=g)
    cuts = [0] + sorted(torch.randint(0, M + 1, (k - 1,), generator=torch.Generator().manual_seed(3)).tolist()) + [M]
    total = torch.zeros(bins, device=DEV, dtype=torch.int32)
    st = torch.zeros(1, device=DEV, dtype=torch.int32)
    for a, b in zip(cuts[:-1], cuts[1:]):
        part = hits[perm[a:b]].contiguous()
        hist = torch.zeros(bins, device=DEV, dtype=torch.int32)
        call("ps_hits_histogram", ptr(part), part.numel(), ptr(hist), bins, ptr(st), stream())
        total += hist
    assert int(st) == 0
    got = torch.zeros(1, device=DEV, dtype=torch.float64)
    call("ps_hits_quantile_from_histogram", ptr(total), bins, M, float(q), ptr(got), stream())
    assert torch.equal(got, want)


@pytest.mark.parametrize("shape", ["c2", "presight16"])
def test_sharded_extractor_of_one_rank_matches_prior_extractor(shape):
    import torch.distributed as dist
    from presight_b200.extract import PriorExtractor, ShardedPriorExtractor
    assert not (dist.is_available() and dist.is_initialized())
    model, _ = c2_model() if shape == "c2" else presight_model()
    n = 20000
    rb = synth_bundle(n, seed=17)
    colors = torch.rand(n, 3, generator=torch.Generator().manual_seed(5)).to(DEV)
    kw = dict(max_range_m=60.0, z_range_m=(-3.0, 12.0), chunk_rays=2500, block_hits=5000, insert_slice=3000)
    ref = PriorExtractor(model, SCALE, **kw)
    ref.add(rb, colors)
    want = ref.finalize()
    ex = ShardedPriorExtractor(model, SCALE, **kw)
    assert ex.world == 1 and ex.rank == 0
    ex.add(rb, colors)
    assert len(ex._blocks) > 1
    got = ex.finalize()
    assert ex.exchanged_bytes == 0
    assert_same_priors(got, want)
