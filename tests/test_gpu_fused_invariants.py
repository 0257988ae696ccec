"""The fused tcgen05 level kernels (csrc/field_tc5_*.cu, csrc/prop_tc5.cu) against themselves on re-composed batches.

The kernels are persistent: each CTA loops over tiles of 128 sample rows (`tile += gridDim.x`), prefetches the next
tile's features, and keeps the weight / bias gradients in tensor memory until the end of the kernel or until the
sub-field changes.  Their structure fixes the right answer of a re-composed batch exactly:

- every per-ray output depends on that ray alone, so a ray's forward outputs and its rows of the feature gradient are
  bit-identical whatever tile, row or CTA it lands in ("exact", torch.equal);
- weight, bias, table and appearance gradients are sums over rays, so they add up over disjoint ray sets, a ray with zero
  upstream gradient adds exactly zero, and one ray in a large batch gives what it gives alone.  Those sums go through fp32
  atomics and tensor-memory accumulation in an order that depends on the batch, so they are compared to fp32 summation
  noise (REORDER) — except for what the ray cannot reach at all, which must be exactly zero.

The small cases are tied to the oracle and to the modular kernels by test_gpu_fused.py / test_gpu_ms.py; these tests run
at sizes where a CTA works through several tiles, reaches its prefetched buffer and changes sub-field."""
import ctypes as C

import pytest
import torch

import oracle as O
import test_gpu_ms
from helpers import rel_err
from test_gpu_fused import _tc5_case, build_single_field_model, make_batch

pytestmark = pytest.mark.gpu
DEV = "cuda"

REORDER = 1e-5          # fp32 sums whose order depends on the batch: atomics, tensor-memory accumulation over tiles
ROWS = 128              # sample rows per tile (kRows)
NUM_SMS = 148           # kNumSMs: the persistent kernels launch at most this many CTAs per resident CTA slot of an SM
MAX_PROP_CTAS = 8       # resident proposal-level CTAs per SM: derived at the first launch, capped at 8 (prop_tc5.cu)
PROP_MS_BWD_CTAS = 4    # resident CTAs per SM of the sub-field proposal backward (prop_tc5.cu launch_ms)
AABB = [-1.0, -1.0, -0.5, 1.0, 1.0, 0.5]
FIELD_OUTS = ("w", "rgb", "acc", "dexp", "sem")


# ------------------------------------------------------------------------------------------------ launch arithmetic
def rays_per_tile(S):
    return ROWS // S


def tiles_of(n, S):
    return -(-n // rays_per_tile(S))


def rays_for_tiles(S, tiles):
    """A batch of `tiles` tiles whose last tile is partial wherever a tile holds more than one ray."""
    rpt = rays_per_tile(S)
    return tiles * rpt - (1 if rpt > 1 else 0)


def field_fwd_grid(ntiles):
    return min(-(-ntiles // 2), NUM_SMS)            # CTAs of the field forward: one per pair of tiles


def field_bwd_grid(ntiles):
    return min(ntiles, NUM_SMS)


def prop_grid(ntiles, ctas_per_sm):
    return min(ntiles, NUM_SMS * ctas_per_sm)


def placement_tiles(ntiles, grids):
    """Tiles to give a one-hot ray: the first, the last, and for each grid size g the last tile of a CTA's first round
    (g - 1) and the first two of its second round (g, g + 1), the ones read from the prefetched buffer."""
    ts = {0, ntiles - 1}
    for g in grids:
        ts |= {g - 1, g, g + 1}
    return sorted(t for t in ts if 0 <= t < ntiles)


def ray_in_tile(t, n, S):
    """A ray of tile t, at a row offset that varies with t; the last tile gets the batch's last ray."""
    rpt = rays_per_tile(S)
    if t == tiles_of(n, S) - 1:
        return n - 1
    return t * rpt + t % rpt


def recompositions(n, S, seed):
    """(name, ray index lists) of re-composed batches: sub-batches cut at tile boundaries, the batch shifted by one ray
    (each ray at another row of its tile) and a permutation."""
    rpt = rays_per_tile(S)
    nt = tiles_of(n, S)
    cuts = [0, rpt * (NUM_SMS + 1), rpt * (nt // 2 + 3), n]
    g = torch.Generator().manual_seed(seed)
    return [("whole-tile sub-batches", [torch.arange(a, b) for a, b in zip(cuts[:-1], cuts[1:])]),
            ("shifted by one ray", [torch.arange(1, n)]),
            ("permutation", [torch.randperm(n, generator=g)])]


def ray_masks(n, seed):
    """Two disjoint ray masks that cover the batch, as float 0/1 columns."""
    a = torch.rand(n, generator=torch.Generator().manual_seed(seed)) < 0.5
    return a.float(), (~a).float()


def reach_mask(corner_rows, table_rows):
    """Table rows a set of points can touch: [P, L, 8] corner rows (ops.hash_indices / oracle.hash_corner_indices)."""
    m = torch.zeros(table_rows, dtype=torch.bool, device=corner_rows.device)
    m[corner_rows.reshape(-1)] = True
    return m


def scaled(G, col):
    """Upstream gradients G (dict of [N, ...] tensors) with row i multiplied by col[i] (0/1: exact)."""
    return {k: v * col.to(v.device).view(-1, *[1] * (v.dim() - 1)) for k, v in G.items()}


def rows_of(G, idx):
    return {k: v[idx.to(v.device)].contiguous() for k, v in G.items()}


# ------------------------------------------------------------------------------------------------ comparisons
def assert_equal_rows(got, want, what):
    assert got.shape == want.shape, f"{what}: shape {tuple(got.shape)} != {tuple(want.shape)}"
    if not torch.equal(got, want):
        bad = (got != want).reshape(got.shape[0], -1).any(dim=1).nonzero().flatten()
        raise AssertionError(f"{what}: {bad.numel()} rows differ (first {bad[:8].tolist()}), max |diff| "
                             f"{float((got - want).abs().max()):.3e}")


def assert_reorder(got, want, what, scale=None):
    """max |got - want| <= REORDER * scale (default: max |want|)."""
    e = rel_err(got, want) if scale is None else float((got.double() - want.double()).abs().max()) / (scale + 1e-30)
    assert e <= REORDER, f"{what}: scale-relative error {e:.3e} > {REORDER:.0e}"


def output_bias_scale(grads, k):
    """The density output's bias gradient is one number, the sum of d raw over every point of the level (or sub-field):
    it cancels heavily, so its fp32 summation-order noise follows the size of the summed terms, not of the sum.  It is
    measured against the larger of itself and its layer's weight gradient (sums of the same d raw times the hidden
    activations).  None for every other gradient."""
    w = "W1" if k == "b1" else k[:-len("bias")] + "weight" if k.endswith("mlp_base.1.layers.1.bias") else None
    if w is None or grads.get(w) is None or grads[k] is None or grads[k].numel() != 1:
        return None
    return max(float(grads[k].abs().max()), float(grads[w].abs().max()))


def assert_zero(t, what):
    assert t is None or not bool(t.any()), f"{what}: {int((t != 0).sum())} non-zero entries, max {float(t.abs().max()):.3e}"


def assert_grads_reorder(got, want, what):
    for k in want:
        g, w = got[k], want[k]
        if g is None or w is None:
            assert_zero(g, f"{what} {k}")
            assert_zero(w, f"{what} {k}")
        else:
            assert_reorder(g, w, f"{what} {k}", output_bias_scale(want, k))


# ------------------------------------------------------------------------------------------------ field level, ray mode
# (S, L, F, A): every S, both kernel instances (L*F <= 32 and 33..48), F in {2, 4}, A in {0, 7, 16}
FIELD_CASES = [(S, L, F, (0, 7, 16)[i % 3]) for i, (S, (L, F)) in enumerate(
    (S, lf) for S in (32, 64, 96, 128) for lf in ((16, 2), (8, 4), (20, 2), (12, 4)))]
FIELD_TILES = 7 * NUM_SMS + 3       # >= 3 tile pairs per CTA in the forward, 7 tiles per CTA in the backward


def _field_ws_bs(c):
    ws = [*c["nets"]["base"][0], *c["nets"]["sem"][0], *c["nets"]["rgb"][0]]
    bs = [*c["nets"]["base"][1], *c["nets"]["sem"][1], *c["nets"]["rgb"][1]]
    return ws, bs


def _field_upstream(n, S, seed):
    g = torch.Generator().manual_seed(seed)
    G = dict(w=torch.randn(n, S, 1, generator=g) * 0.05, rgb=torch.randn(n, 3, generator=g),
             acc=torch.randn(n, 1, generator=g), dexp=torch.randn(n, 1, generator=g), sem=torch.randn(n, 64, generator=g))
    return {k: v.to(DEV) for k, v in G.items()}


def _field_fwd(c, idx):
    """ps_field_level_fwd on the rays `idx` -> (per-ray outputs, tminmax, (sel, feat, app) for the backward)."""
    from presight_b200 import fused
    ws, bs = _field_ws_bs(c)
    i = idx.to(DEV)
    app = None if c["app"] is None else c["app"].detach()[i].contiguous()
    with torch.no_grad():
        _, sel, feat, w, rgb, acc, dexp, dthr, sem, tmm = fused.tc5_field_forward(
            c["o"][i].contiguous(), c["d"][i].contiguous(), c["eu"][i].contiguous(), app, c["table"].detach(), c["aabb"],
            True, c["grid"], [x.detach() for x in ws], [x.detach() for x in bs], c["A"], 0.5)
    return dict(w=w, rgb=rgb, acc=acc, dexp=dexp, dthr=dthr, sem=sem), tmm, (sel, feat, app)


def _field_bwd_abi(c, idx, G):
    """ps_field_level_bwd at the C-ABI (as _FieldLevelTc5.backward calls it) on the rays `idx`; G: upstream gradients of
    those rays, None = not given (NULL).  -> (dfeat [L, N, S, F], dapp, dW, dB)."""
    from presight_b200 import ops
    from presight_b200._lib import call, host_field_net, ptr
    out, _, (sel, feat, app) = _field_fwd(c, idx)
    N, S, A = len(idx), c["eu"].shape[1] - 1, c["A"]
    i = idx.to(DEV)
    ws, bs = [[x.detach() for x in t] for t in _field_ws_bs(c)]
    zs = ops.zeros_like_many([*ws, *bs])
    dW, dB = zs[:8], zs[8:]
    dapp = torch.zeros(N, A, device=DEV) if A else None
    net = host_field_net(ws, bs, A, dW, dB)
    dfeat = torch.full_like(feat, float("nan"))       # an entry the kernel does not write shows up as NaN
    gw = None if G["w"] is None else G["w"].reshape(N, S).contiguous()
    # ptr() keeps only an address: every tensor the kernel reads must stay referenced until it is enqueued, or the
    # caching allocator may hand its block to the next temporary of the argument list
    eu, d = c["eu"][i].contiguous(), c["d"][i].contiguous()
    call("ps_field_level_bwd", C.byref(net), ptr(feat), c["grid"].L, c["grid"].F, ptr(sel), ptr(eu), ptr(d), ptr(app),
         N, S, ptr(out["acc"]), ptr(out["dexp"]), ptr(gw), ptr(G["rgb"]), ptr(G["acc"]), ptr(G["dexp"]), ptr(G["sem"]),
         ptr(dfeat), ptr(dapp), torch.cuda.current_stream().cuda_stream)
    return dfeat.view(c["grid"].L, N, S, c["grid"].F), dapp, dW, dB


def _field_grads(c, idx, G, zeros_for_absent=False):
    """_FieldLevelTc5 (autograd) on the rays `idx`; G: upstream gradients of those rays, a missing / None entry = an
    output the loss does not use (or, zeros_for_absent, one given an explicit zero gradient).  -> name -> gradient."""
    from presight_b200 import fused
    ws, bs = _field_ws_bs(c)
    i = idx.to(DEV)
    app = None if c["app"] is None else c["app"].detach()[i].contiguous().requires_grad_(True)
    out = fused._FieldLevelTc5.apply(c["o"][i].contiguous(), c["d"][i].contiguous(), c["eu"][i].contiguous(), app,
                                     c["table"], c["aabb"], True, c["grid"], 0.5, *ws, *bs)
    outs = dict(zip(("w", "rgb", "acc", "dexp", "dthr", "sem", "tmm"), out))
    keys = [k for k in FIELD_OUTS if G.get(k) is not None or zeros_for_absent]
    grads_out = [G[k] if G.get(k) is not None else torch.zeros_like(outs[k]) for k in keys]
    names = ["table"] + [f"W{j}" for j in range(8)] + [f"b{j}" for j in range(8)] + (["app"] if app is not None else [])
    leaves = [c["table"], *ws, *bs] + ([app] if app is not None else [])
    gs = torch.autograd.grad([outs[k] for k in keys], leaves, grads_out, allow_unused=True)
    return dict(zip(names, gs))


@pytest.mark.parametrize("S,L,F,A", FIELD_CASES)
def test_field_forward_rays_are_independent(S, L, F, A):
    """ps_field_level_fwd: every per-ray output is bit-identical in sub-batches cut at tile boundaries, shifted by one row
    and permuted; the batch's tminmax is the min / max over the sub-batches'."""
    n = rays_for_tiles(S, FIELD_TILES)
    assert field_fwd_grid(tiles_of(n, S)) == NUM_SMS and tiles_of(n, S) >= 3 * 2 * NUM_SMS
    c = _tc5_case(n, S, A, L, F, seed=S + L)
    full, tmm, _ = _field_fwd(c, torch.arange(n))
    for name, parts in recompositions(n, S, seed=S):
        tmms = []
        for idx in parts:
            got, tm, _ = _field_fwd(c, idx)
            tmms.append(tm)
            for k in ("w", "rgb", "acc", "dexp", "dthr", "sem"):
                assert_equal_rows(got[k], full[k][idx.to(DEV)], f"{name}: {k}")
        lo = torch.stack([t[0] for t in tmms]).min()
        hi = torch.stack([t[1] for t in tmms]).max()
        assert torch.equal(torch.stack([lo, hi]), tmm), f"{name}: tminmax"


@pytest.mark.parametrize("S,L,F,A", FIELD_CASES)
def test_field_backward_feature_gradient_is_per_ray(S, L, F, A):
    """ps_field_level_bwd: a ray's rows of dfeat are bit-identical under the same re-compositions; its appearance
    gradient (atomics over the ray's warps) agrees to fp32 summation order."""
    n = rays_for_tiles(S, FIELD_TILES)
    c = _tc5_case(n, S, A, L, F, seed=S + L + 1)
    G = _field_upstream(n, S, seed=S)
    dfeat, dapp, _, _ = _field_bwd_abi(c, torch.arange(n), G)
    assert bool(dfeat.abs().amax() > 0)
    for name, parts in recompositions(n, S, seed=S + 1):
        for idx in parts:
            df, da, _, _ = _field_bwd_abi(c, idx, rows_of(G, idx))
            i = idx.to(DEV)
            assert_equal_rows(df.transpose(0, 1), dfeat[:, i].transpose(0, 1), f"{name}: dfeat")
            if A:
                assert_reorder(da, dapp[i], f"{name}: dapp")


# (S, L, F, A) of the gradient tests: both kernel instances, a partial last tile in each
FIELD_GRAD_CASES = [(64, 16, 2, 16), (32, 12, 4, 7)]


@pytest.mark.parametrize("S,L,F,A", FIELD_GRAD_CASES)
def test_field_gradients_are_tile_local_and_additive(S, L, F, A):
    """_FieldLevelTc5 backward: zero upstream gradient gives exactly zero gradients; gradients of disjoint ray sets add
    up; one ray with upstream gradient in a large batch gives what it gives alone, in the first and the last tile and
    where a CTA reaches its second tile, and nothing outside that ray's reach."""
    from presight_b200 import fused, ops
    n = rays_for_tiles(S, FIELD_TILES)
    ntiles = tiles_of(n, S)
    grid = field_bwd_grid(ntiles)
    assert ntiles >= 3 * grid and n % rays_per_tile(S) != 0
    c = _tc5_case(n, S, A, L, F, seed=3)
    G = _field_upstream(n, S, seed=4)
    everyone = torch.arange(n)
    full = _field_grads(c, everyone, G)
    assert all(bool(v.any()) for v in full.values())
    for k, v in _field_grads(c, everyone, scaled(G, torch.zeros(n))).items():
        assert_zero(v, f"zero upstream gradient: {k}")
    ma, mb = ray_masks(n, seed=5)
    ga, gb = _field_grads(c, everyone, scaled(G, ma)), _field_grads(c, everyone, scaled(G, mb))
    assert_grads_reorder({k: ga[k] + gb[k] for k in full}, full, "disjoint rays")
    T = c["table"].shape[0]
    for t in placement_tiles(ntiles, [grid]):
        r = ray_in_tile(t, n, S)
        hot = torch.zeros(n)
        hot[r] = 1.0
        batch = _field_grads(c, everyone, scaled(G, hot))
        alone = _field_grads(c, torch.tensor([r]), rows_of(G, torch.tensor([r])))
        what = f"ray {r} in tile {t} of {ntiles} (grid {grid})"
        for k in alone:
            if k == "app":
                assert_reorder(batch[k][r:r + 1], alone[k], f"{what}: dapp")
                others = torch.ones(n, dtype=torch.bool, device=DEV)
                others[r] = False
                assert_zero(batch[k][others], f"{what}: other rays' dapp")
            else:
                assert_reorder(batch[k], alone[k], f"{what}: {k}")
        x01, _ = fused._ray_points(c["o"][r:r + 1], c["d"][r:r + 1], c["eu"][r:r + 1], c["aabb"], True)
        corners, _ = ops.hash_indices(x01, c["grid"].scalings, c["grid"].log2_T)
        assert_zero(batch["table"][~reach_mask(corners, T)], f"{what}: table rows outside its corners")


@pytest.mark.parametrize("absent", [("w", "acc", "dexp", "sem"), ("dexp",), ("w",), ("w", "rgb", "acc", "dexp")],
                         ids=["only-rgb", "no-depth", "no-weights", "only-semantics"])
def test_field_absent_upstream_gradients_equal_zero_ones(absent):
    """Upstream gradients autograd does not produce reach ps_field_level_bwd as NULL: the result equals that of explicit
    zero gradients — dfeat exactly at the C-ABI, parameter / table / appearance gradients to fp32 summation order."""
    S, A = 64, 16
    n = rays_for_tiles(S, 3 * NUM_SMS + 1)
    c = _tc5_case(n, S, A, 16, 2, seed=8)
    G = _field_upstream(n, S, seed=9)
    missing = {k: (None if k in absent else v) for k, v in G.items()}
    zero = {k: (torch.zeros_like(v) if k in absent else v) for k, v in G.items()}
    everyone = torch.arange(n)
    df_n, dapp_n, dW_n, dB_n = _field_bwd_abi(c, everyone, missing)
    df_z, dapp_z, dW_z, dB_z = _field_bwd_abi(c, everyone, zero)
    assert bool(df_z.any())
    assert torch.equal(df_n, df_z), "dfeat with NULL upstream gradients"
    assert_reorder(dapp_n, dapp_z, "dapp")
    for j in range(8):
        assert_reorder(dW_n[j], dW_z[j], f"dW{j}")
        assert_reorder(dB_n[j], dB_z[j], f"db{j}")
    assert_grads_reorder(_field_grads(c, everyone, missing), _field_grads(c, everyone, G | {k: None for k in absent},
                                                                          zeros_for_absent=True), "autograd")


# ------------------------------------------------------------------------------------------------ proposal and density levels
PROP_CASES = [(16, 1, 32, 12), (16, 2, 64, 8), (64, 1, 128, 16), (64, 2, 96, 5)]      # (H, F, S, L)
PROP_TILES = 3 * NUM_SMS * MAX_PROP_CTAS + 5       # >= 3 tiles per CTA whatever the resident CTAs per SM


def _prop_case(n, S, L, F, H, seed, hidden_out=1):
    from presight_b200 import fused
    g = torch.Generator().manual_seed(seed)
    log2T = 14
    scal = tuple(O.hash_scalings(L, 16, 1024).tolist())
    table = ((torch.rand(L << log2T, F, generator=g) * 2 - 1) * 2.0).to(DEV).requires_grad_(True)
    dims = (L * F, H, hidden_out)
    ws = [(torch.randn(dims[i + 1], dims[i], generator=g) / dims[i] ** 0.5).to(DEV).requires_grad_(True) for i in range(2)]
    bs = [(torch.randn(dims[i + 1], generator=g) * 0.1).to(DEV).requires_grad_(True) for i in range(2)]
    o = ((torch.rand(n, 3, generator=g) - 0.5) * torch.tensor([1.0, 1.0, 0.1])).to(DEV)
    d = torch.nn.functional.normalize(torch.randn(n, 3, generator=g), dim=-1).to(DEV)
    eu = (torch.rand(n, S + 1, generator=g) * 0.05 + 0.001).cumsum(-1).to(DEV)
    return dict(o=o, d=d, eu=eu, table=table, params=[ws[0], bs[0], ws[1], bs[1]], grid=fused.GridMeta(scal, log2T, F))


def _prop_weights(p, idx):
    from presight_b200 import fused
    i = idx.to(DEV)
    return fused._PropLevelTc5.apply(p["o"][i].contiguous(), p["d"][i].contiguous(), p["eu"][i].contiguous(), p["table"],
                                     AABB, True, p["grid"], None, *p["params"])


def _prop_grads(p, idx, gw):
    w = _prop_weights(p, idx)
    gs = torch.autograd.grad(w, [p["table"], *p["params"]], gw)
    return dict(zip(("table", "W0", "b0", "W1", "b1"), gs))


@pytest.mark.parametrize("H,F,S,L", PROP_CASES)
def test_prop_forward_rays_are_independent(H, F, S, L):
    """ps_prop_level_fwd: a ray's weights are bit-identical under the re-compositions."""
    n = rays_for_tiles(S, PROP_TILES)
    p = _prop_case(n, S, L, F, H, seed=H + F)
    with torch.no_grad():
        full = _prop_weights(p, torch.arange(n))
        for name, parts in recompositions(n, S, seed=H):
            for idx in parts:
                assert_equal_rows(_prop_weights(p, idx), full[idx.to(DEV)], f"{name}: weights")


# (F, L, S): the density heads' instances F in {1, 2, 4} x K0 in {16, 32, 48} that L <= 32 levels reach, every S
DENSITY_CASES = [(F, L, (32, 64, 96, 128)[i % 4]) for i, (F, L) in enumerate(
    ((1, 12), (1, 24), (2, 8), (2, 16), (2, 20), (4, 4), (4, 8), (4, 12)))]


@pytest.mark.parametrize("F,L,S", DENSITY_CASES)
def test_density_forward_rays_are_independent(F, L, S):
    """ps_density_level_fwd (the main field's density head on the proposal kernels): per-ray weights bit-identical under
    the re-compositions."""
    from presight_b200._lib import call, host_prop_net, host_floats, ptr
    n = rays_for_tiles(S, PROP_TILES)
    p = _prop_case(n, S, L, F, 64, seed=F + L, hidden_out=80)       # base1 is [80, 64]: row 0 / bias[0] are the density
    net = host_prop_net([x.detach() for x in p["params"][0::2]], [x.detach() for x in p["params"][1::2]])
    g = p["grid"]

    def weights(idx):
        i = idx.to(DEV)
        w = torch.full((len(idx), S), float("nan"), device=DEV)      # unwritten weights show up as NaN
        o, d, eu = (p[k][i].contiguous() for k in ("o", "d", "eu"))   # referenced until the kernel is enqueued
        call("ps_density_level_fwd", C.byref(net), ptr(o), ptr(d), ptr(eu), len(idx), S, host_floats(AABB), 1,
             ptr(p["table"].detach()), host_floats(g.scalings), g.L, g.F, g.log2_T, ptr(w),
             torch.cuda.current_stream().cuda_stream)
        return w
    full = weights(torch.arange(n))
    assert bool((full > 0).any())
    for name, parts in recompositions(n, S, seed=L):
        for idx in parts:
            assert_equal_rows(weights(idx), full[idx.to(DEV)], f"{name}: weights")


@pytest.mark.parametrize("H,F,S,L", PROP_CASES)
def test_prop_gradients_are_tile_local_and_additive(H, F, S, L):
    """_PropLevelTc5 backward: zero upstream gradient -> exactly zero; disjoint ray sets add up; a one-hot ray gives what
    it gives alone, placed around every grid size the resident-CTA count can produce (1..8 per SM), and touches no table
    row outside its samples' corners."""
    from presight_b200 import fused, ops
    n = rays_for_tiles(S, PROP_TILES)
    ntiles = tiles_of(n, S)
    assert ntiles >= 3 * prop_grid(ntiles, MAX_PROP_CTAS)
    p = _prop_case(n, S, L, F, H, seed=H * F + S)
    gw = (torch.randn(n, S, 1, generator=torch.Generator().manual_seed(S)) * 0.1).to(DEV)
    everyone = torch.arange(n)
    full = _prop_grads(p, everyone, gw)
    assert all(bool(v.any()) for v in full.values())
    for k, v in _prop_grads(p, everyone, torch.zeros_like(gw)).items():
        assert_zero(v, f"zero upstream gradient: {k}")
    ma, mb = ray_masks(n, seed=S)
    ga, gb = _prop_grads(p, everyone, gw * ma.to(DEV).view(-1, 1, 1)), _prop_grads(p, everyone, gw * mb.to(DEV).view(-1, 1, 1))
    assert_grads_reorder({k: ga[k] + gb[k] for k in full}, full, "disjoint rays")
    grids = [prop_grid(ntiles, c) for c in range(1, MAX_PROP_CTAS + 1)]
    T = p["table"].shape[0]
    for t in placement_tiles(ntiles, grids):
        r = ray_in_tile(t, n, S)
        hot = torch.zeros(n, 1, 1, device=DEV)
        hot[r] = 1.0
        batch = _prop_grads(p, everyone, gw * hot)
        alone = _prop_grads(p, torch.tensor([r]), gw[r:r + 1].contiguous())
        what = f"ray {r} in tile {t} of {ntiles}"
        for k in alone:
            assert_reorder(batch[k], alone[k], f"{what}: {k}", output_bias_scale(alone, k))
        x01, _ = fused._ray_points(p["o"][r:r + 1], p["d"][r:r + 1], p["eu"][r:r + 1], AABB, True)
        corners, _ = ops.hash_indices(x01, p["grid"].scalings, p["grid"].log2_T)
        assert_zero(batch["table"][~reach_mask(corners, T)], f"{what}: table rows outside its corners")


# ------------------------------------------------------------------------------------------------ sub-field mode
MS_S = 64
# >= 3 tiles per CTA of the sub-field proposal backward (the kernel with the largest grid) once routed
MS_RAYS = -(-3 * NUM_SMS * PROP_MS_BWD_CTAS * ROWS // MS_S)


@pytest.fixture(scope="module")
def ms_case():
    """16 routed sub-fields (test_gpu_ms.build), MS_RAYS rays with 64 samples each and per-ray appearance."""
    model, _, host = test_gpu_ms.build(MS_RAYS)
    g = torch.Generator().manual_seed(11)
    o, d = host["origins"].to(DEV), host["directions"].to(DEV)
    eu = (torch.sort(torch.rand(MS_RAYS, MS_S + 1, generator=g), dim=1).values * 40.0 + 0.01).to(DEV)
    app = torch.randn(MS_RAYS, 16, generator=g).to(DEV)
    return model, o, d, eu, app


def _contract(router):
    return router.fields[0].spatial_distortion is not None


def _sub_field_of(name):
    return int(name.split(".")[1]) if name.startswith("fields.") else None


def _ms_rays(rt, grid, S):
    """Rays to place a one-hot gradient on, from a level's routing: one with a sample in the first and in the last live
    tile, around `grid` (a CTA's first and second round) and in the first tile where a CTA changes sub-field."""
    tile_sf, perm = rt.tile_sf.cpu().long(), rt.perm.cpu().long()
    live = int((tile_sf != 255).sum())
    tiles = {0, live - 1} | {t for t in (grid - 1, grid, grid + 1) if t < live}
    switch = [t for t in range(grid, live) if tile_sf[t] != tile_sf[t - grid]]
    assert switch, "no CTA changes sub-field: the batch is too small"
    tiles.add(switch[0])
    rays = {}
    for t in sorted(tiles):
        pts = perm[t * ROWS:(t + 1) * ROWS]
        pts = pts[pts >= 0]
        assert pts.numel(), f"tile {t} holds no point"
        rays.setdefault(int(pts[len(pts) // 2]) // S, t)
    return rays


def _ms_reach(rt1, grid_meta, tables):
    """Per sub-field: the table-row mask one ray's samples can touch (its routing rt1), or None if none routes there."""
    from presight_b200 import ops
    rows = (rt1.perm >= 0).nonzero().flatten()
    sfs = rt1.tile_sf.long()[rows // ROWS]
    reach = {}
    for k in range(len(tables)):
        rk = rows[sfs == k]
        if rk.numel():
            corners, _ = ops.hash_indices(rt1.x01[rk], grid_meta.scalings, grid_meta.log2_T)
            reach[k] = reach_mask(corners, tables[k].shape[0])
    return reach


def _check_one_hot_ms(batch, alone, reach, r, what):
    for k, a in alone.items():
        b, sf = batch[k], _sub_field_of(k)
        if k == "app":
            assert_reorder(b[r:r + 1], a, f"{what}: dapp")
            assert_zero(torch.cat([b[:r], b[r + 1:]]), f"{what}: other rays' dapp")
        elif sf not in reach:
            assert_zero(b, f"{what}: {k} (sub-field {sf} not reached)")
            assert_zero(a, f"{what}: {k} alone (sub-field {sf} not reached)")
        else:
            assert_reorder(b, a, f"{what}: {k}", output_bias_scale(alone, k))
            if k.endswith("hash_table"):
                assert_zero(b[~reach[sf]], f"{what}: {k} rows outside its corners")


def test_sub_field_forward_rays_are_independent(ms_case):
    """Sub-field mode (routing + ps_field_level_fwd_ms / ps_prop_level_fwd_ms + compositing): a ray's outputs are
    bit-identical alone, in a permuted batch and in the batch shifted by one ray."""
    model, o, d, eu, app = ms_case
    from presight_b200 import fused
    field, prop = model.field, model.proposal_networks[0]
    assert len(field.fields) == test_gpu_ms.NF and field._ms_meta() is not None and prop._ms_meta() is not None

    def run(idx):
        i = idx.to(DEV)
        with torch.no_grad():
            w, rgb, acc, dexp, dthr, sem, _ = field.fused_level(o[i], d[i], eu[i], app[i], 0.5)
            pw = prop.level_weights(o[i], d[i], eu[i])
        return dict(w=w, rgb=rgb, acc=acc, dexp=dexp, dthr=dthr, sem=sem, prop_w=pw)
    full = run(torch.arange(MS_RAYS))
    rt = fused.route_points(field.centroids, field._aabbs_host(), _contract(field), o, d, eu)
    assert len(set(rt.tile_sf.cpu().tolist()) - {255}) >= 4, "the rays should reach several sub-fields"
    singles = [torch.tensor([r]) for r in _ms_rays(rt, field_bwd_grid(rt.rows // ROWS), MS_S)]
    g = torch.Generator().manual_seed(2)
    for name, idx in [("permutation", torch.randperm(MS_RAYS, generator=g)), ("shifted by one ray", torch.arange(1, MS_RAYS))] \
            + [(f"ray {int(s)} alone", s) for s in singles]:
        got = run(idx)
        for k, v in got.items():
            assert_equal_rows(v, full[k][idx.to(DEV)], f"{name}: {k}")


def _ms_field_grads(model, ms_case, idx, G):
    """model.field.fused_level on the rays `idx` with upstream gradients G (rows of idx; a missing output is not used by
    the loss) -> parameter name -> gradient, and "app"."""
    _, o, d, eu, app = ms_case
    i = idx.to(DEV)
    a = app[i].contiguous().requires_grad_(True)
    out = dict(zip(("w", "rgb", "acc", "dexp", "dthr", "sem", "tmm"), model.field.fused_level(o[i], d[i], eu[i], a, 0.5)))
    names, params = zip(*model.field.named_parameters())
    keys = [k for k in FIELD_OUTS if G.get(k) is not None]
    gs = torch.autograd.grad([out[k] for k in keys], [*params, a], [G[k] for k in keys], allow_unused=True)
    return dict(zip([*names, "app"], gs))


def _ms_prop_grads(prop, ms_case, idx, gw):
    _, o, d, eu, _ = ms_case
    i = idx.to(DEV)
    w = prop.level_weights(o[i], d[i], eu[i])
    names, params = zip(*prop.named_parameters())
    return dict(zip(names, torch.autograd.grad(w, params, gw, allow_unused=True)))


def test_sub_field_gradients_are_tile_local_and_additive(ms_case):
    """Sub-field mode backward (ps_field_level_bwd_ms, ps_prop_level_bwd_ms and their scatters): zero upstream gradient
    -> exactly zero; disjoint ray sets add up; a one-hot ray — in the first and last tiles, around the grid and where a
    CTA flushes one sub-field's gradients and starts the next — gives what it gives alone, and exactly zero in every
    sub-field none of its samples routes to and in every table row outside its samples' corners."""
    from presight_b200 import fused
    model, o, d, eu, app = ms_case
    field, prop = model.field, model.proposal_networks[0]
    n, S = MS_RAYS, MS_S
    everyone = torch.arange(n)
    G = _field_upstream(n, S, seed=12)
    gw = G["w"]
    full = _ms_field_grads(model, ms_case, everyone, G)
    pfull = _ms_prop_grads(prop, ms_case, everyone, gw)
    reached = {_sub_field_of(k) for k, v in full.items() if v is not None and bool(v.any())} - {None}
    assert len(reached) >= 4
    for k, v in _ms_field_grads(model, ms_case, everyone, scaled(G, torch.zeros(n))).items():
        assert_zero(v, f"zero upstream gradient: field {k}")
    for k, v in _ms_prop_grads(prop, ms_case, everyone, torch.zeros_like(gw)).items():
        assert_zero(v, f"zero upstream gradient: proposal {k}")
    ma, mb = ray_masks(n, seed=13)
    ga, gb = _ms_field_grads(model, ms_case, everyone, scaled(G, ma)), _ms_field_grads(model, ms_case, everyone, scaled(G, mb))
    add = lambda x, y: None if x is None and y is None else (0 if x is None else x) + (0 if y is None else y)  # noqa: E731
    assert_grads_reorder({k: add(ga[k], gb[k]) for k in full}, full, "disjoint rays: field")
    pa = _ms_prop_grads(prop, ms_case, everyone, gw * ma.to(DEV).view(-1, 1, 1))
    pb = _ms_prop_grads(prop, ms_case, everyone, gw * mb.to(DEV).view(-1, 1, 1))
    assert_grads_reorder({k: add(pa[k], pb[k]) for k in pfull}, pfull, "disjoint rays: proposal")

    fgrid, ftables = field._ms_meta(), [f.mlp_base_grid.hash_table for f in field.fields]
    pgrid, ptables = prop._ms_meta(), [f.encoding.hash_table for f in prop.fields]
    p_aabbs = [list(f.aabb_host()) for f in prop.fields]
    rt = fused.route_points(field.centroids, field._aabbs_host(), _contract(field), o, d, eu)
    prt = fused.route_points(prop.centroids, p_aabbs, _contract(prop), o, d, eu)
    cases = [("field", r, t) for r, t in _ms_rays(rt, field_bwd_grid(rt.rows // ROWS), S).items()] + \
            [("proposal", r, t) for r, t in _ms_rays(prt, prop_grid(prt.rows // ROWS, PROP_MS_BWD_CTAS), S).items()]
    for level, r, t in cases:
        one = torch.tensor([r])
        hot = torch.zeros(n)
        hot[r] = 1.0
        what = f"{level}: ray {r} (a sample in tile {t})"
        if level == "field":
            batch = _ms_field_grads(model, ms_case, everyone, scaled(G, hot))
            alone = _ms_field_grads(model, ms_case, one, rows_of(G, one))
            rt1 = fused.route_points(field.centroids, field._aabbs_host(), _contract(field), o[r:r + 1], d[r:r + 1], eu[r:r + 1])
            _check_one_hot_ms(batch, alone, _ms_reach(rt1, fgrid, ftables), r, what)
        else:
            batch = _ms_prop_grads(prop, ms_case, everyone, gw * hot.to(DEV).view(-1, 1, 1))
            alone = _ms_prop_grads(prop, ms_case, one, gw[r:r + 1].contiguous())
            rt1 = fused.route_points(prop.centroids, p_aabbs, _contract(prop), o[r:r + 1], d[r:r + 1], eu[r:r + 1])
            _check_one_hot_ms(batch, alone, _ms_reach(rt1, pgrid, ptables), r, what)


@pytest.mark.parametrize("absent", [("w", "acc", "dexp", "sem"), ("dexp",), ("w",), ("w", "rgb", "acc", "dexp")],
                         ids=["only-rgb", "no-depth", "no-weights", "only-semantics"])
def test_sub_field_absent_upstream_gradients_equal_zero_ones(ms_case, absent):
    """Sub-field mode through model.field.fused_level: a loss on a subset of the outputs gives the gradients of the full
    loss with zero weight on the other outputs (the wrapper fills in what autograd did not produce)."""
    model = ms_case[0]
    n = MS_RAYS
    everyone = torch.arange(n)
    G = _field_upstream(n, MS_S, seed=14)
    subset = _ms_field_grads(model, ms_case, everyone, {k: (None if k in absent else v) for k, v in G.items()})
    zeros = _ms_field_grads(model, ms_case, everyone, {k: (torch.zeros_like(v) if k in absent else v) for k, v in G.items()})
    assert any(v is not None and bool(v.any()) for v in zeros.values())
    assert_grads_reorder(subset, zeros, "subset vs zero-weighted loss")


# ------------------------------------------------------------------------------------------------ side-stream proposal backward
def test_side_stream_proposal_backward_matches_in_order(monkeypatch):
    """One training step of the single-field model with the interlevel loss: the proposal backwards on the side stream
    (handed off through ops.publish_grad_event / pop_grad_event) give the gradients of the in-order schedule."""
    from presight_b200 import fused, losses, ops
    n = 2048
    model, _ = build_single_field_model("b200", samples=(64, 32, 32))      # proposal levels on _PropLevelTc5
    model.train()
    bundle, jit, tgt, _ = make_batch(n, seed=6)
    pop = ops.pop_grad_event
    handed_off = [0]

    def counting_pop(t, key):
        ev = pop(t, key)
        handed_off[0] += ev is not None
        return ev
    monkeypatch.setattr(ops, "pop_grad_event", counting_pop)

    def step(overlap):
        prev = fused.set_overlap_prop_bwd(overlap)
        try:
            model.zero_grad(set_to_none=True)
            model.proposal_sampler._step = 0
            out = model(bundle(), jitters=jit)
            loss = ((out["rgb"] - tgt["rgb"]) ** 2).mean() + 0.5 * ((out["semantics"] - tgt["sem"]) ** 2).mean() \
                + losses.interlevel_loss(out["weights_list"], [rs.sp_bins for rs in out["ray_samples_list"]])
            loss.backward()
            torch.cuda.synchronize()
        finally:
            fused.set_overlap_prop_bwd(prev)
        return {k: p.grad.clone() for k, p in model.named_parameters() if k.startswith("proposal_networks.")}
    in_order = step(False)
    assert handed_off[0] == 0
    side = step(True)
    assert handed_off[0] == len(model.proposal_networks), f"{handed_off[0]} proposal backwards ran on the side stream"
    assert in_order.keys() == side.keys() and len(side) >= 10
    for k in in_order:
        assert bool(in_order[k].any()), k
        assert_reorder(side[k], in_order[k], k)
