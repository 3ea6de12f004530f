"""Differential fuzz of the data-shard iterator's host side (SURVEY §8 a-11) against the unmodified reference
(`dmlcloud/util/data.py`).  oracle/gen_golden.py ran the reference on the same seeded random cases and stored its answers
in tests/golden/shard_fuzz.json: the length and a SHA-256 digest of each index list (the full lists would not fit a small
fixture).  Index lists are integers: every comparison is exact."""
import hashlib

import numpy as np
import torch

from conftest import load_json


def digest(values):
    """Length and SHA-256 of an integer sequence, the form the reference's answers are stored in."""
    values = list(values)
    return [len(values), hashlib.sha256(np.asarray(values, dtype=np.int64).tobytes()).hexdigest()]


def digest_tensors(tensors):
    """Count and SHA-256 over the shapes, dtypes and bytes of a list of tensors."""
    h = hashlib.sha256()
    for t in tensors:
        h.update(repr((tuple(t.shape), str(t.dtype))).encode())
        h.update(t.contiguous().numpy().tobytes())
    return [len(tensors), h.hexdigest()]


def shard_index_cases():
    rng = np.random.RandomState(5)
    for _ in range(400):
        n, world = int(rng.randint(0, 5000)), int(rng.randint(1, 9))
        rank, seed = int(rng.randint(world)), int(rng.randint(0, 2**31 - 1))
        yield (n, rank, world), dict(shuffle=bool(rng.randint(2)), even_shards=bool(rng.randint(2)), seed=seed)


def chunk_and_sequence_cases():
    rng = np.random.RandomState(6)
    for _ in range(200):
        n, world, chunk = int(rng.randint(1, 3000)), int(rng.randint(1, 9)), int(rng.randint(1, 64))
        rank, seed = int(rng.randint(world)), int(rng.randint(0, 2**31 - 1))
        yield (n, chunk, rank, world), dict(shuffle=bool(rng.randint(2)), even_shards=bool(rng.randint(2)), seed=seed)


def dataset_epoch_cases():
    rng = np.random.RandomState(7)
    for _ in range(60):
        n, world = int(rng.randint(1, 500)), int(rng.randint(1, 9))
        rank, seed, epoch = int(rng.randint(world)), int(rng.randint(0, 10**6)), int(rng.randint(0, 20))
        yield (n, epoch), dict(shuffle=bool(rng.randint(2)), even_shards=bool(rng.randint(2)), seed=seed, rank=rank,
                               world_size=world)


def interleave_cases():
    rng = np.random.RandomState(8)
    for _ in range(40):
        k, batch, width = int(rng.randint(1, 6)), int(rng.randint(1, 5)), int(rng.randint(1, 4))
        batch *= k  # the reference requires the batch size to be divisible by num_batches
        n_batches = k * int(rng.randint(1, 4))
        g = torch.Generator().manual_seed(int(rng.randint(10**6)))
        yield k, [torch.randn(batch, width, generator=g) for _ in range(n_batches)]


def run_shard_indices(fn):
    return [digest(fn(*args, **kw)) for args, kw in shard_index_cases()]


def run_chunks_and_sequences(chunk_and_shard_indices, shard_sequence):
    out = []
    for (n, chunk, rank, world), kw in chunk_and_sequence_cases():
        out.append(digest(chunk_and_shard_indices(n, chunk, rank, world, **kw)))
        out.append(digest(shard_sequence(list(range(1000, 1000 + n)), rank, world, **kw)))
    return out


def run_dataset_epochs(ShardedSequenceDataset):
    out = []
    for (n, epoch), kw in dataset_epoch_cases():
        ds = ShardedSequenceDataset(list(range(n)), **kw)
        ds.set_epoch(epoch)
        out.append(digest(iter(ds)))
    return out


def run_interleave(interleave_batches):
    return [digest_tensors(list(interleave_batches(iter(data), k))) for k, data in interleave_cases()]


def check(got, want, cases):
    assert len(got) == len(want)
    for case, g, w in zip(cases, got, want):
        assert g == w, case


def test_shard_indices_random_cases():
    from dmlcloud_b200.util.data import shard_indices

    check(run_shard_indices(shard_indices), load_json('shard_fuzz.json')['shard_indices'], list(shard_index_cases()))


def test_chunked_sharding_and_sequences_random_cases():
    from dmlcloud_b200.util.data import chunk_and_shard_indices, shard_sequence

    cases = [(c, what) for c in chunk_and_sequence_cases() for what in ('chunk_and_shard_indices', 'shard_sequence')]
    check(run_chunks_and_sequences(chunk_and_shard_indices, shard_sequence),
          load_json('shard_fuzz.json')['chunks_and_sequences'], cases)


def test_sharded_sequence_dataset_epochs():
    from dmlcloud_b200.util.data import ShardedSequenceDataset

    check(run_dataset_epochs(ShardedSequenceDataset), load_json('shard_fuzz.json')['dataset_epochs'],
          list(dataset_epoch_cases()))


def test_interleave_batches_random_cases():
    from dmlcloud_b200.util.data import interleave_batches

    check(run_interleave(interleave_batches), load_json('shard_fuzz.json')['interleave'],
          [(k, len(data)) for k, data in interleave_cases()])
