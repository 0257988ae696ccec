"""Worker of tests/test_gpu_sharded_extract_multi.py, launched with torchrun on >= 2 GPUs of one box (NCCL).

Every rank builds the same seeded model and the same rays, adds its share to a ShardedPriorExtractor and calls
finalize(dst); rank dst also runs a single-GPU PriorExtractor on all the rays, and the two results must agree as
assert_same_priors states it.  Cases (argv[1], comma-separated):

  c2, presight16   an even split of the rays over the ranks
  uneven           rank 0 adds 70 % of the rays, the result lands on the last rank
  idle             rank 0 (the destination) adds no ray at all
  rounds           small store blocks and a 75 / 25 split: the ranks hold different numbers of blocks, so the exchange
                   has several rounds, some of them empty on one side
  skewed           80 % of the rays are copies of 16 rays: most hits share a few voxels
"""
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

SCALE = 0.05
KW = dict(max_range_m=60.0, z_range_m=(-3.0, 12.0))
CASES = {
    "c2": dict(shape="c2", first=None),
    "presight16": dict(shape="presight16", first=None),
    "uneven": dict(shape="c2", first=0.7, dst=-1),
    "idle": dict(shape="c2", first=0.0),
    "rounds": dict(shape="c2", first=0.75, chunk_rays=1000, block_hits=1500),
    "skewed": dict(shape="c2", first=None, skew=True),
}


def share(n, first, rank, world):
    """[lo, hi) of rank's rays: rank 0 takes `first` of them (None: an even split), the others split the rest."""
    from presight_b200.parallel import shard_range
    if first is None:
        return shard_range(n, rank, world)
    k = int(round(first * n))
    if rank == 0:
        return 0, k
    lo, hi = shard_range(n - k, rank - 1, world - 1)
    return k + lo, k + hi


def run_case(name, rank, world):
    from test_gpu_extract import c2_model, presight_model, synth_bundle
    from test_gpu_tile_extract import assert_same_priors
    from presight_b200.cameras.rays import RayBundle
    from presight_b200.extract import PriorExtractor, ShardedPriorExtractor
    cfg = CASES[name]
    dst = cfg.get("dst", 0) % world
    model, _ = c2_model() if cfg["shape"] == "c2" else presight_model()
    n = 40000
    rb = synth_bundle(n, seed=23)
    if cfg.get("skew"):
        g = torch.Generator().manual_seed(8)
        idx = torch.cat([torch.randint(0, 16, (int(0.8 * n),), generator=g), torch.arange(16, n - int(0.8 * n) + 16)])
        idx = idx[torch.randperm(n, generator=g)].to(rb.origins.device)
        rb = RayBundle(origins=rb.origins[idx].contiguous(), directions=rb.directions[idx].contiguous())
    colors = torch.rand(n, 3, generator=torch.Generator().manual_seed(6)).to(rb.origins.device)
    sizes = dict(chunk_rays=cfg.get("chunk_rays", 4096), block_hits=cfg.get("block_hits", 8192), insert_slice=5000)
    lo, hi = share(n, cfg["first"], rank, world)
    ex = ShardedPriorExtractor(model, SCALE, **sizes, **KW)
    if hi > lo:
        ex.add(RayBundle(origins=rb.origins[lo:hi], directions=rb.directions[lo:hi]), colors[lo:hi])
    blocks = torch.tensor([len(ex._blocks)], device=rb.origins.device)
    per_rank = [torch.zeros_like(blocks) for _ in range(world)]
    dist.all_gather(per_rank, blocks)
    per_rank = [int(b) for b in per_rank]
    got = ex.finalize(dst)
    sent = torch.tensor([ex.exchanged_bytes], device=rb.origins.device)
    dist.all_reduce(sent)
    if name == "idle":
        assert per_rank[0] == 0
    if name == "rounds":
        assert len(set(per_rank)) > 1 and max(per_rank) > 2, per_rank
    if rank != dst:
        assert got is None
        return
    ref = PriorExtractor(model, SCALE, **sizes, **KW)
    ref.add(rb, colors)
    want = ref.finalize()
    assert_same_priors(got, want)
    if cfg.get("skew"):
        assert int(want["hits"].max()) > 1000, int(want["hits"].max())
    print(f"SHARDED {name} ok: world {world}, dst {dst}, blocks per rank {per_rank}, stored hits {ref.n_hits}, voxels "
          f"{got['n_voxels']}, kept {got['hits'].numel()}, max hits {int(want['hits'].max())}, thr {float(got['hit_thr'])}, "
          f"exchanged {int(sent)} B", flush=True)


def main():
    dist.init_process_group("nccl")
    rank, world = dist.get_rank(), dist.get_world_size()
    torch.cuda.set_device(int(os.environ["LOCAL_RANK"]))
    for name in sys.argv[1].split(","):
        try:
            run_case(name, rank, world)
        except Exception as e:                    # report and go on: every case is its own test
            print(f"SHARDED {name} FAILED on rank {rank}: {type(e).__name__}: {e}", flush=True)
        dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
