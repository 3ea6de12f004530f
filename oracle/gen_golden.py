"""ORACLE — TEST INFRASTRUCTURE ONLY.  Golden-vector generator.

Runs the UNMODIFIED reference (/root/reference, importable only in the build container, with the three dependency shims
under oracle/shims/) on torch.distributed/gloo CPU and writes small fixtures to tests/golden/:

  shard_indices.json     reference util/data.py:11-30 known answers (incl. shuffled, seeds, ShardedSequenceDataset epochs)
  metrics_w{1,2,4}.json  a scripted MetricTracker session (script + every rank's resulting histories), metrics.py
  grads_*.npz            per-rank local gradients (inputs) and the DDP(gloo)-reduced gradients (reference output)
  train_w{1,2,4,8}.json  a short TrainValStage + DDP(gloo) MNIST-CNN run on synthetic data: full tracker.histories
  train_clip_w{1,2}.json the same run with gradient_clip() != 0;  train_sched_w1.json with a StepLR scheduler
  shard_fuzz.json        digests of util/data.py's answers to tests/test_shard_fuzz_vs_reference.py's random cases
  metric_fuzz_w{1..4}.json  every rank's histories after tests/test_metric_fuzz_vs_reference.py's random sessions

Usage (build container only):  python oracle/gen_golden.py
Nothing on the GPU box may call this: /root/reference does not exist there; tests read the committed fixtures.
"""
import json
import os
import sys
import tempfile
from pathlib import Path

HERE = Path(__file__).resolve().parent
REPO = HERE.parent
GOLD = REPO / 'tests' / 'golden'
sys.path.insert(0, str(HERE / 'shims'))
sys.path.insert(1, '/root/reference')

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402
import torch.multiprocessing as mp  # noqa: E402


# ----------------------------------------------------------------------------------------------------------------------
# helpers
# ----------------------------------------------------------------------------------------------------------------------
def _spawn(fn, world, *args):
    """Run fn(rank, world, initfile, outdir, *args) on `world` gloo ranks; returns outdir Path contents loader."""
    tmp = tempfile.mkdtemp(prefix='dmlb_gold_')
    initfile = os.path.join(tmp, 'init')
    mp.spawn(fn, args=(world, initfile, tmp) + args, nprocs=world, join=True)
    return Path(tmp)


def _init(rank, world, initfile):
    torch.set_num_threads(1)
    dist.init_process_group('gloo', init_method=f'file://{initfile}', rank=rank, world_size=world)


def enc(v):
    """history entry -> JSON."""
    if v is None:
        return None
    if isinstance(v, torch.Tensor):
        return {'dtype': str(v.dtype).replace('torch.', ''), 'shape': list(v.shape), 'data': v.flatten().tolist()}
    if isinstance(v, (int, float, str, bool)):
        return {'py': v}
    raise TypeError(type(v))


# ----------------------------------------------------------------------------------------------------------------------
# 1. shard indices
# ----------------------------------------------------------------------------------------------------------------------
def gen_shards():
    from dmlcloud.util.data import shard_indices, ShardedSequenceDataset

    cases = []
    for n, world in [(10, 2), (10, 3), (11, 2), (20, 2), (64, 8), (1000, 4), (1001, 8)]:
        for rank in range(world):
            for shuffle in (False, True):
                for even in (False, True):
                    for seed in (0, 7):
                        cases.append({
                            'n': n, 'rank': rank, 'world': world, 'shuffle': shuffle, 'even_shards': even, 'seed': seed,
                            'out': shard_indices(n, rank, world, shuffle=shuffle, even_shards=even, seed=seed),
                        })
    heads = []
    for n, seed in [(10, 0), (1000, 7), (60000, 3), (60000, 0), (70000, 12345)]:
        full = shard_indices(n, 0, 1, shuffle=True, even_shards=False, seed=seed)
        heads.append({'n': n, 'seed': seed, 'head': full[:16], 'tail': full[-4:],
                      'checksum': int(np.dot(np.asarray(full, dtype=np.int64) % 1000003, np.arange(n) % 997))})
    epochs = []
    for epoch in (0, 1, 5):
        for rank in range(4):
            ds = ShardedSequenceDataset(list(range(100, 150)), shuffle=True, seed=11, rank=rank, world_size=4)
            ds.set_epoch(epoch)
            epochs.append({'epoch': epoch, 'rank': rank, 'world': 4, 'seed': 11, 'base': 100, 'len': 50,
                           'out': list(iter(ds))})
    (GOLD / 'shard_indices.json').write_text(json.dumps({'cases': cases, 'heads': heads, 'epochs': epochs}))
    print('shard_indices.json', len(cases), 'cases')


# ----------------------------------------------------------------------------------------------------------------------
# 2. metric tracker session
# ----------------------------------------------------------------------------------------------------------------------
def metric_script(world, seed=1234):
    """A deterministic session touching every branch of metrics.py: all reductions, scalar + shaped values with `dim`,
    int64 counters, local-only metrics, un-reduced metrics, late registration (None back-fill), an epoch in which a
    metric gets no values (-> None), prefix reduce + strict/non-strict."""
    rng = np.random.RandomState(seed)
    S = []

    def vals(shape, dtype='float32', lo=-3, hi=3):
        out = []
        for _ in range(world):
            if dtype == 'int64':
                out.append(rng.randint(lo, hi + 1, size=shape).tolist())
            else:
                out.append(rng.uniform(lo, hi, size=shape).astype(np.float32).tolist())
        return out

    S.append(['register', 'plain', None, None, True])
    for red in ('MEAN', 'SUM', 'MIN', 'MAX'):
        S.append(['register', f'g/{red}', red, None, True])
        S.append(['register', f'l/{red}', red, None, False])
    S.append(['register', 'cnt', 'SUM', None, True])
    S.append(['register', 'shape/min12', 'MIN', [1, 2], True])
    S.append(['register', 'shape/sum2', 'SUM', [2], True])
    S.append(['register', 'shape/mean0', 'MEAN', [0], True])
    S.append(['register', 'shape/maxall', 'MAX', None, True])
    for epoch in range(1, 5):
        n_steps = 5 + epoch
        for step in range(n_steps):
            for red in ('MEAN', 'SUM', 'MIN', 'MAX'):
                S.append(['track', f'g/{red}', vals(()), 'float32'])
                S.append(['track', f'l/{red}', vals(()), 'float32'])
            S.append(['track', 'cnt', [[1][0]] * world, 'int64'])
            if epoch != 2:  # epoch 2: shaped metrics get no values on any rank -> None
                S.append(['track', 'shape/min12', vals((2, 2, 3)), 'float32'])
                S.append(['track', 'shape/sum2', vals((2, 2, 3)), 'float32'])
                S.append(['track', 'shape/mean0', vals((4, 3)), 'float32'])
                S.append(['track', 'shape/maxall', vals((3, 5), 'int64', -50, 50), 'int64'])
        S.append(['track_plain', 'plain', epoch * 10])
        if epoch == 2:
            S.append(['register', 'late/mean', 'MEAN', None, True])
            S.append(['track', 'late/mean', vals(()), 'float32'])
            S.append(['reduce_all', 'g/', True])
            S.append(['reduce_all', 'g/', False])
        if epoch == 3:
            S.append(['track', 'late/mean', vals(()), 'float32'])
            S.append(['track', 'late/mean', vals(()), 'float32'])
        S.append(['next_epoch'])
    return S


def _metrics_worker(rank, world, initfile, outdir, script):
    _init(rank, world, initfile)
    from dmlcloud.metrics import MetricTracker, Reduction

    tracker = MetricTracker()
    for op in script:
        if op[0] == 'register':
            _, name, red, dim, glob = op
            tracker.register_metric(name, None if red is None else Reduction[red], dim, glob)
        elif op[0] == 'track':
            _, name, per_rank, dtype = op
            tracker.track(name, torch.tensor(per_rank[rank], dtype=getattr(torch, dtype)))
        elif op[0] == 'track_plain':
            tracker.track(op[1], op[2])
        elif op[0] == 'reduce_all':
            tracker.reduce_all(prefix=op[1], strict=op[2])
        elif op[0] == 'next_epoch':
            tracker.next_epoch()
    out = {'epoch': tracker.epoch, 'histories': {k: [enc(v) for v in h] for k, h in tracker.histories.items()}}
    Path(outdir, f'rank{rank}.json').write_text(json.dumps(out))
    dist.destroy_process_group()


def gen_metrics():
    for world in (1, 2, 4):
        script = metric_script(world)
        out = _spawn(_metrics_worker, world, script)
        ranks = [json.loads((out / f'rank{r}.json').read_text()) for r in range(world)]
        (GOLD / f'metrics_w{world}.json').write_text(json.dumps({'world': world, 'script': script, 'ranks': ranks}))
        print(f'metrics_w{world}.json', len(script), 'ops')


# ----------------------------------------------------------------------------------------------------------------------
# 3. gradient buckets: local grads in, DDP(gloo)-reduced grads out
# ----------------------------------------------------------------------------------------------------------------------
def make_model(kind):
    from torch import nn

    torch.manual_seed(0)
    if kind == 'linear64':
        return nn.Linear(64, 64), (16, 64), 64
    if kind == 'mnist_cnn':  # examples/mnist.py:27-36
        return nn.Sequential(
            nn.Conv2d(1, 16, 3, padding=1), nn.ReLU(), nn.MaxPool2d(2),
            nn.Conv2d(16, 16, 3, padding=1), nn.ReLU(), nn.MaxPool2d(2),
            nn.Flatten(), nn.Linear(784, 10),
        ), (8, 1, 28, 28), 10
    raise ValueError(kind)


def _grads_worker(rank, world, initfile, outdir, kind, steps):
    import copy

    from torch.nn.parallel import DistributedDataParallel

    _init(rank, world, initfile)
    model, in_shape, n_cls = make_model(kind)
    shadow = copy.deepcopy(model)
    ddp = DistributedDataParallel(model, broadcast_buffers=False)  # exactly what pipeline.py:74 builds on CPU
    loss_fn = torch.nn.CrossEntropyLoss()
    g = torch.Generator().manual_seed(1000 + rank)
    local, reduced = [], []
    for _ in range(steps):
        x = torch.randn(in_shape, generator=g)
        y = torch.randint(0, n_cls, (in_shape[0],), generator=g)
        for m in (ddp, shadow):
            m.zero_grad()
            loss_fn(m(x), y).backward()
        local.append(torch.cat([p.grad.flatten() for p in shadow.parameters()]).numpy().copy())
        reduced.append(torch.cat([p.grad.flatten() for p in model.parameters()]).numpy().copy())
    np.save(os.path.join(outdir, f'local{rank}.npy'), np.stack(local))
    if rank == 0:
        np.save(os.path.join(outdir, 'reduced.npy'), np.stack(reduced))
    dist.destroy_process_group()


def gen_grads():
    for kind, worlds, steps in (('linear64', (1, 2, 3, 4, 8), 2), ('mnist_cnn', (2, 3), 2)):
        for world in worlds:
            out = _spawn(_grads_worker, world, kind, steps)
            local = np.stack([np.load(out / f'local{r}.npy') for r in range(world)], axis=1)  # [S, W, N]
            reduced = np.load(out / 'reduced.npy')  # [S, N]
            np.savez_compressed(GOLD / f'grads_{kind}_w{world}.npz', local=local, reduced=reduced)
            err = np.abs(local.astype(np.float64).mean(1) - reduced).max() / np.abs(reduced).max()
            print(f'grads_{kind}_w{world}.npz', local.shape, f'ref-vs-fp64 rel err {err:.2e}')


# ----------------------------------------------------------------------------------------------------------------------
# 4. short TrainValStage run (reference stage.py:290-335 + pipeline.py) on synthetic MNIST-shaped data
# ----------------------------------------------------------------------------------------------------------------------
TRAIN_STEPS, VAL_STEPS, EPOCHS, BATCH = 6, 2, 2, 32


def synthetic_batches(seed, steps, batch=BATCH):
    g = torch.Generator().manual_seed(seed)
    return [(torch.randn(batch, 1, 28, 28, generator=g), torch.randint(0, 10, (batch,), generator=g))
            for _ in range(steps)]


CLIP_NORM = 0.05  # small enough that the coefficient is < 1 on most steps of the synthetic run


def _train_worker(rank, world, initfile, outdir, variant='plain'):
    """variant: 'plain' | 'clip' (gradient_clip() = CLIP_NORM, stage.py:256-285) | 'sched' (StepLR stepped per epoch,
    stage.py:316-318, three epochs so that two different learning rates are applied)."""
    _init(rank, world, initfile)
    from dmlcloud.pipeline import TrainingPipeline
    from dmlcloud.stage import TrainValStage

    class MNISTStage(TrainValStage):
        def pre_stage(self):
            self.pipeline.register_dataset('train', synthetic_batches(100 + rank, TRAIN_STEPS), verbose=False)
            self.pipeline.register_dataset('val', synthetic_batches(200 + rank, VAL_STEPS), verbose=False)
            model, _, _ = make_model('mnist_cnn')
            self.pipeline.register_model('cnn', model, verbose=False)
            optimizer = torch.optim.Adam(model.parameters(), lr=1e-3)
            scheduler = torch.optim.lr_scheduler.StepLR(optimizer, step_size=1, gamma=0.5) if variant == 'sched' else None
            self.pipeline.register_optimizer('adam', optimizer, scheduler)
            self.loss = torch.nn.CrossEntropyLoss()

        def gradient_clip(self):
            return CLIP_NORM if variant == 'clip' else 0.0

        def step(self, batch):
            img, target = batch
            output = self.pipeline.models['cnn'](img)
            loss = self.loss(output, target)
            self.track_reduce('accuracy', (output.argmax(1) == target).float().mean())
            return loss

    import contextlib
    import io

    pipeline = TrainingPipeline(name='golden')
    stage = MNISTStage()
    pipeline.append_stage(stage, max_epochs=EPOCHS + (1 if variant == 'sched' else 0))
    with contextlib.redirect_stdout(io.StringIO()):
        pipeline.run()
    hist = {k: [enc(v) for v in h] for k, h in pipeline.tracker.histories.items()}
    final = torch.cat([p.detach().flatten() for p in pipeline.models['cnn'].parameters()])
    out = {'tracker_epoch': pipeline.tracker.epoch, 'stage_epoch': stage.current_epoch, 'histories': hist,
           'param_sum': float(final.double().sum()), 'param_abs_sum': float(final.double().abs().sum())}
    Path(outdir, f'rank{rank}.json').write_text(json.dumps(out))
    dist.destroy_process_group()


def gen_train():
    runs = [('plain', w, f'train_w{w}.json') for w in (1, 2, 4, 8)]
    runs += [('clip', w, f'train_clip_w{w}.json') for w in (1, 2)] + [('sched', 1, 'train_sched_w1.json')]
    for variant, world, fname in runs:
        out = _spawn(_train_worker, world, variant)
        ranks = [json.loads((out / f'rank{r}.json').read_text()) for r in range(world)]
        meta = {'world': world, 'train_steps': TRAIN_STEPS, 'val_steps': VAL_STEPS,
                'epochs': EPOCHS + (1 if variant == 'sched' else 0), 'batch': BATCH,
                'train_seed': '100+rank', 'val_seed': '200+rank', 'init_seed': 0, 'optimizer': 'Adam(lr=1e-3)'}
        if variant == 'clip':
            meta['gradient_clip'] = CLIP_NORM
        if variant == 'sched':
            meta['scheduler'] = 'StepLR(step_size=1, gamma=0.5)'
        (GOLD / fname).write_text(json.dumps({'meta': meta, 'ranks': ranks}))
        print(fname, {k: v[-1] for k, v in ranks[0]['histories'].items() if 'loss' in k})


# ----------------------------------------------------------------------------------------------------------------------
# 5. the reference's answers to the seeded random cases of the differential fuzz tests
# ----------------------------------------------------------------------------------------------------------------------
FUZZ_SEEDS = {1: range(60), 2: range(2000, 2012), 3: range(3000, 3012), 4: range(4000, 4010)}  # the tests' seeds


def _fuzz_tests():
    sys.path.insert(0, str(REPO / 'tests'))
    import test_metric_fuzz_vs_reference
    import test_shard_fuzz_vs_reference

    return test_shard_fuzz_vs_reference, test_metric_fuzz_vs_reference


def _fuzz_metrics_worker(rank, world, initfile, outdir, seeds):
    _init(rank, world, initfile)
    from dmlcloud.metrics import MetricTracker, Reduction

    _, T = _fuzz_tests()
    sessions = {}
    for seed in seeds:
        script = T.random_session(seed, world)
        tracker = MetricTracker()
        T.replay(tracker, Reduction, script, rank)
        sessions[str(seed)] = {'script_sha256': T.script_digest(script), 'epoch': tracker.epoch,
                               'histories': {k: [enc(v) for v in h] for k, h in tracker.histories.items()}}
    Path(outdir, f'rank{rank}.json').write_text(json.dumps(sessions))
    dist.destroy_process_group()


def gen_fuzz():
    from dmlcloud.util import data

    S, _ = _fuzz_tests()
    out = {'shard_indices': S.run_shard_indices(data.shard_indices),
           'chunks_and_sequences': S.run_chunks_and_sequences(data.chunk_and_shard_indices, data.shard_sequence),
           'dataset_epochs': S.run_dataset_epochs(data.ShardedSequenceDataset),
           'interleave': S.run_interleave(data.interleave_batches)}
    (GOLD / 'shard_fuzz.json').write_text(json.dumps(out))
    print('shard_fuzz.json', {k: len(v) for k, v in out.items()})
    for world, seeds in FUZZ_SEEDS.items():
        out = _spawn(_fuzz_metrics_worker, world, list(seeds))
        ranks = [json.loads((out / f'rank{r}.json').read_text()) for r in range(world)]
        sessions = {}
        for seed in map(str, seeds):
            assert len({ranks[r][seed]['script_sha256'] for r in range(world)}) == 1
            sessions[seed] = {'script_sha256': ranks[0][seed]['script_sha256'],
                              'ranks': [{k: ranks[r][seed][k] for k in ('epoch', 'histories')} for r in range(world)]}
        (GOLD / f'metric_fuzz_w{world}.json').write_text(json.dumps({'world': world, 'sessions': sessions}))
        print(f'metric_fuzz_w{world}.json', len(sessions), 'sessions')


if __name__ == '__main__':
    if not Path('/root/reference/dmlcloud').is_dir():
        sys.exit('gen_golden.py needs /root/reference (build container only)')
    GOLD.mkdir(parents=True, exist_ok=True)
    which = sys.argv[1:] or ['shards', 'metrics', 'grads', 'train', 'fuzz']
    if 'shards' in which:
        gen_shards()
    if 'metrics' in which:
        gen_metrics()
    if 'grads' in which:
        gen_grads()
    if 'train' in which:
        gen_train()
    if 'fuzz' in which:
        gen_fuzz()
