"""CPU tests of the sharding the sequence-only DeepCNN branch uses: `shard_job(..., alpha=0)`, LPT bins on a cost linear in the
sequence length (the convolution works per 128-residue tile; there is no L^2 stage)."""
import numpy as np
import pytest

from metagenomic_deepfri_b200 import distributed, sharding


@pytest.mark.parametrize("world", [1, 2, 3, 8])
def test_linear_cost_shards_cover_bound_and_balance(world):
    rng = np.random.default_rng(world)
    lengths = np.clip(np.exp(rng.normal(np.log(250.0), 0.6, size=20_000)), 50, 1000).astype(np.int64)
    shards = distributed.shard_job(lengths, world, max_proteins=1000, max_residues=200_000, alpha=0.0)
    assert len(shards) == world
    allidx = np.concatenate([c for chunks in shards for c in chunks])
    assert np.array_equal(np.sort(allidx), np.arange(len(lengths)))          # every index exactly once
    for chunks in shards:
        for c in chunks:
            assert 1 <= len(c) <= 1000 and (lengths[c].sum() <= 200_000 or len(c) == 1)
            assert np.all(np.diff(c) > 0)
    loads = np.array([sum(int(lengths[c].sum()) for c in chunks) for chunks in shards], np.float64)
    # greedy list scheduling: no bin exceeds the mean by more than the largest item; at this size that is well under 1 %
    assert loads.max() <= loads.mean() + lengths.max()
    assert loads.max() / loads.mean() <= 1.01


def test_alpha_zero_is_the_residue_balance():
    """With alpha = 0 the bins balance residues, not the GCN's quadratic cost: the same LPT as bins over plain lengths."""
    lengths = np.random.default_rng(3).integers(1, 3000, 5000)
    got = distributed.shard_job(lengths, 4, max_proteins=1 << 30, max_residues=1 << 40, alpha=0.0)
    want = sharding.lpt_bins(lengths, 4, alpha=0.0)
    assert all(np.array_equal(np.concatenate(g), w) for g, w in zip(got, want))
    default = distributed.shard_job(lengths, 4, max_proteins=1 << 30, max_residues=1 << 40)
    assert any(not np.array_equal(np.concatenate(g), np.concatenate(d)) for g, d in zip(got, default))
