"""Differential fuzz of the metric path (SURVEY §8 a-4..a-8) against the unmodified reference.

Seeded random sessions — random metric sets (all reductions, `dim` subsets, int64 and fp32 values, rank-local metrics,
un-reduced metrics), random step counts, epochs in which a metric gets no value, late registration, prefix reduces — are
replayed on this repo's MetricTracker (host logic) over oracle/slab_oracle.py (the bit-level restatement of the device slab
the GPU tests compare libdmlb with), at world size 1, 2 and 3 (gloo), and compared with what the reference's own
MetricTracker computed for the same sessions: oracle/gen_golden.py replayed them on the reference and stored every rank's
resulting histories in tests/golden/metric_fuzz_w{1,2,3,4}.json (the script's SHA-256 beside them pins the session).
This pins host logic + slab oracle to the reference far beyond the fixed golden sessions: the GPU parity tests then carry
that over to the kernels.

Tolerances (SURVEY §8d): MIN / MAX, integer results, None patterns, dtypes, shapes, epochs: exact; fp32 MEAN / SUM: rtol 1e-5,
atol 1e-6 (the reference reduces a stacked fp32 tensor, the slab accumulates in fp64 and rounds once).
"""
import functools
import hashlib
import json
from pathlib import Path
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from conftest import decode_entry, load_json
from helpers import init_gloo, spawn

REDUCTIONS = ('MEAN', 'SUM', 'MIN', 'MAX')


def script_digest(script):
    return hashlib.sha256(json.dumps(script).encode()).hexdigest()


@functools.lru_cache(maxsize=None)
def reference_sessions(world):
    return load_json(f'metric_fuzz_w{world}.json')['sessions']


def reference_tracker(world, seed, rank, script):
    """The reference MetricTracker's state after `script` on `rank`, as stored by oracle/gen_golden.py."""
    session = reference_sessions(world)[str(seed)]
    assert session['script_sha256'] == script_digest(script), ('the session generator changed', world, seed)
    state = session['ranks'][rank]

    def decode(e):
        v = decode_entry(e)
        return torch.from_numpy(v) if isinstance(v, np.ndarray) else v

    return SimpleNamespace(epoch=state['epoch'],
                           histories={name: [decode(e) for e in h] for name, h in state['histories'].items()})


def random_session(seed, world):
    """[op, ...] with per-rank values; ops: register / track / track_plain / reduce_all / next_epoch (as gen_golden.py)."""
    rng = np.random.RandomState(seed)
    metrics, script = {}, []

    def new_metric(tag):
        red = REDUCTIONS[rng.randint(4)]
        shape = tuple(int(s) for s in rng.randint(1, 4, size=rng.randint(0, 4)))
        integer = red != 'MEAN' and rng.rand() < 0.3  # (mean of an int64 tensor raises in torch, reference included)
        dim = None
        if shape and rng.rand() < 0.6:
            k = rng.randint(1, len(shape) + 1)
            dim = sorted(int(d) for d in rng.choice(len(shape), size=k, replace=False))
        name = f'{("a", "b")[rng.randint(2)]}/{tag}'
        metrics[name] = {'shape': shape, 'int': integer, 'p_skip': (0.0, 0.0, 0.5)[rng.randint(3)]}
        script.append(['register', name, red, dim, bool(rng.rand() < 0.75)])
        return name

    for i in range(rng.randint(2, 7)):
        new_metric(f'm{i}')
    script.append(['register', 'plain', None, None, True])
    n_epochs = rng.randint(2, 5)
    for epoch in range(n_epochs):
        if epoch == 1 and rng.rand() < 0.7:
            new_metric('late')  # registered after an epoch has closed: its history is back-filled with None
        skipped = {n for n, m in metrics.items() if rng.rand() < m['p_skip']}  # no value on ANY rank this epoch -> None
        for _ in range(rng.randint(1, 6)):
            for name, m in metrics.items():
                if name in skipped:
                    continue
                if m['int']:
                    per_rank = [rng.randint(-40, 41, size=m['shape']).tolist() for _ in range(world)]
                else:
                    per_rank = [rng.uniform(-3, 3, size=m['shape']).astype(np.float32).tolist() for _ in range(world)]
                script.append(['track', name, per_rank, 'int64' if m['int'] else 'float32'])
        if rng.rand() < 0.8:
            script.append(['track_plain', 'plain', int(rng.randint(100))])
        if rng.rand() < 0.5:
            script.append(['reduce_all', 'a/', True])
            if rng.rand() < 0.5:
                script.append(['reduce_all', 'a/', False])  # non-strict: already reduced metrics are left alone
        script.append(['next_epoch'])
    return script


def replay(tracker, Reduction, script, rank, device=None):
    for op in script:
        if op[0] == 'register':
            tracker.register_metric(op[1], None if op[2] is None else Reduction[op[2]], op[3], op[4])
        elif op[0] == 'track':
            value = torch.tensor(op[2][rank], dtype=getattr(torch, op[3]))
            tracker.track(op[1], value if device is None else value.to(device))
        elif op[0] == 'track_plain':
            tracker.track(op[1], op[2])
        elif op[0] == 'reduce_all':
            tracker.reduce_all(prefix=op[1], strict=op[2])
        else:
            tracker.next_epoch()


def compare(want_tracker, got_tracker, script, seed, exact=False):
    kinds = {op[1]: op[2] for op in script if op[0] == 'register'}
    assert got_tracker.epoch == want_tracker.epoch, seed
    assert list(got_tracker.histories) == list(want_tracker.histories), seed
    for name, want_hist in want_tracker.histories.items():
        got_hist = got_tracker.histories[name]
        assert len(got_hist) == len(want_hist), (seed, name)
        for epoch, (want, got) in enumerate(zip(want_hist, got_hist)):
            where = (seed, name, epoch)
            if want is None or not isinstance(want, torch.Tensor):
                assert got == want and type(got) is type(want), where
                continue
            assert isinstance(got, torch.Tensor), where
            got = got.cpu()
            assert got.dtype == want.dtype and got.shape == want.shape, (where, got.dtype, want.dtype, got.shape, want.shape)
            want = want.cpu()
            if exact or not want.dtype.is_floating_point or kinds[name] in ('MIN', 'MAX'):
                assert torch.equal(got, want), (where, got, want)
            else:
                np.testing.assert_allclose(got.numpy(), want.numpy(), rtol=1e-5, atol=1e-6, err_msg=str(where))


def run_seeds(seeds, world, rank, device=None, comm=None):
    """device=None: this repo's MetricTracker over the slab oracle (CPU).  device=cuda: the product — libdmlb's device slab
    (and `comm`, the peer communicator, at world > 1) — checked against the reference AND, bit for bit, against the slab
    oracle."""
    from dmlcloud_b200.metrics import MetricTracker, Reduction
    from oracle.slab_oracle import OracleSlab

    checked = 0
    for seed in seeds:
        script = random_session(seed, world)
        want = reference_tracker(world, seed, rank, script)
        restated = MetricTracker()
        restated.bind(slab=OracleSlab())
        replay(restated, Reduction, script, rank)
        compare(want, restated, script, seed)
        if device is not None:
            product = MetricTracker()
            product.bind(device=device, comm=comm, group=None)
            replay(product, Reduction, script, rank, device=device)
            compare(want, product, script, seed)
            compare(restated, product, script, seed, exact=True)
        checked += sum(len(h) for h in want.histories.values())
    return checked


def test_random_sessions_match_the_installed_reference_w1():
    import torch.distributed as dist

    from dmlcloud_b200.util.distributed import deinitialize_torch_distributed, init_process_group_dummy

    init_process_group_dummy()
    try:
        assert dist.get_world_size() == 1
        assert run_seeds(range(60), 1, 0) > 500  # history entries compared
    finally:
        deinitialize_torch_distributed()


def _worker(rank, world, initfile, outdir, first_seed, n_seeds):
    init_gloo(rank, world, initfile)
    import torch.distributed as dist

    checked = run_seeds(range(first_seed, first_seed + n_seeds), world, rank)
    Path(outdir, f'ok{rank}.json').write_text(json.dumps({'checked': checked}))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize('world', [2, 3])
def test_random_sessions_match_the_installed_reference_over_gloo(world):
    out = spawn(_worker, world, 1000 * world, 12, timeout=600)
    counts = [json.loads((out / f'ok{r}.json').read_text())['checked'] for r in range(world)]
    assert len(set(counts)) == 1 and counts[0] > 100
