"""Host-side helpers of test_gpu_fused_invariants.py on the CPU at tiny sizes: batch sizes from the kernels' launch
arithmetic, one-hot placements, re-compositions, ray masks, and corner-reach sets against the oracle's hash backward."""
import pytest
import torch

import oracle as O
import test_gpu_fused_invariants as T


@pytest.mark.parametrize("S", [32, 64, 96, 128])
def test_field_batches_reach_the_tiles_they_are_sized_for(S):
    n = T.rays_for_tiles(S, T.FIELD_TILES)
    nt = T.tiles_of(n, S)
    assert nt == T.FIELD_TILES
    assert T.field_fwd_grid(nt) == T.NUM_SMS and nt >= 3 * 2 * T.NUM_SMS          # >= 3 tile pairs per forward CTA
    assert T.field_bwd_grid(nt) == T.NUM_SMS and nt >= 3 * T.NUM_SMS
    assert (n % T.rays_per_tile(S) != 0) == (T.rays_per_tile(S) > 1)               # a partial last tile where possible
    for t in T.placement_tiles(nt, [T.field_bwd_grid(nt)]):
        assert T.ray_in_tile(t, n, S) // T.rays_per_tile(S) == t
    assert T.ray_in_tile(nt - 1, n, S) == n - 1


@pytest.mark.parametrize("H,F,S,L", T.PROP_CASES)
def test_prop_batches_cover_every_resident_cta_count(H, F, S, L):
    n = T.rays_for_tiles(S, T.PROP_TILES)
    nt = T.tiles_of(n, S)
    grids = [T.prop_grid(nt, c) for c in range(1, T.MAX_PROP_CTAS + 1)]
    assert nt >= 3 * max(grids)
    tiles = T.placement_tiles(nt, grids)
    assert {0, nt - 1} <= set(tiles) and all({g - 1, g, g + 1} <= set(tiles) for g in grids)
    assert all(T.ray_in_tile(t, n, S) // T.rays_per_tile(S) == t for t in tiles)


def test_sub_field_batch_gives_three_tiles_per_proposal_backward_cta():
    assert T.MS_RAYS * T.MS_S // T.ROWS >= 3 * T.NUM_SMS * T.PROP_MS_BWD_CTAS


@pytest.mark.parametrize("S", [32, 128])
def test_recompositions_are_whole_tile_cuts_shifts_and_permutations(S):
    n = T.rays_for_tiles(S, T.FIELD_TILES)                    # index tensors only
    parts = dict(T.recompositions(n, S, seed=1))
    cuts = parts["whole-tile sub-batches"]
    assert torch.equal(torch.cat(cuts), torch.arange(n)) and all(int(c[0]) % T.rays_per_tile(S) == 0 for c in cuts)
    assert torch.equal(parts["shifted by one ray"][0], torch.arange(1, n))
    assert torch.equal(torch.sort(parts["permutation"][0]).values, torch.arange(n))


def test_ray_masks_split_the_batch_and_scaling_is_exact():
    a, b = T.ray_masks(200, seed=3)
    assert torch.equal(a + b, torch.ones(200)) and 0 < int(a.sum()) < 200
    G = {"w": torch.randn(4, 3, 1), "rgb": torch.randn(4, 3)}
    col = torch.tensor([0.0, 1.0, 0.0, 1.0])
    sa, sb = T.scaled(G, col), T.scaled(G, 1 - col)
    for k in G:
        assert torch.equal(sa[k] + sb[k], G[k]) and not sa[k][0].any()
    assert torch.equal(T.rows_of(G, torch.tensor([3, 1]))["rgb"], G["rgb"][[3, 1]])


def test_reach_mask_holds_every_row_the_hash_backward_touches():
    g = torch.Generator().manual_seed(0)
    L, log2T, F = 8, 10, 2
    s = O.hash_scalings(L, 16, 512)
    x = torch.rand(5, 3, generator=g)
    table = (torch.rand(L << log2T, F, generator=g) * 2 - 1).requires_grad_(True)
    y = O.hash_encode(x, O.HashGrid(table, s, log2T))
    y.backward(torch.randn_like(y))
    corners, _ = O.hash_corner_indices(x, s, log2T)
    reach = T.reach_mask(corners, table.shape[0])
    touched = table.grad.abs().sum(1) > 0
    assert bool(touched.any()) and not bool((touched & ~reach).any())


def test_output_bias_scale_applies_to_one_number_biases_only():
    grads = {"W1": torch.full((1, 16), 2.0), "b1": torch.tensor([0.5]),
             "fields.3.mlp_base.1.layers.1.weight": torch.full((1, 16), 3.0),
             "fields.3.mlp_base.1.layers.1.bias": torch.tensor([0.1])}
    assert T.output_bias_scale(grads, "b1") == 2.0
    assert T.output_bias_scale(grads, "fields.3.mlp_base.1.layers.1.bias") == 3.0
    assert T.output_bias_scale(grads, "W1") is None
    wide = {"W1": torch.ones(80, 64), "b1": torch.ones(80)}             # the field's base layer: compared as it is
    assert T.output_bias_scale(wide, "b1") is None
