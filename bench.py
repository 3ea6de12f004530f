#!/usr/bin/env python
"""bench.py — samples/sec of the data-parallel training step through dmlcloud_b200 (BASELINE.json metric).

    python bench.py --gpus 1 --steps 200 --warmup 20                       # native arm, one GPU
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
           bench.py --gpus N --steps K --warmup W                          # N ranks, one per GPU
    python bench.py --impl reference --gpus N --steps K --warmup W         # the reference's own CPU/gloo path
    python bench.py --workload resnet18 ...                                # BASELINE config 4 instead of config 2/3

A "step" = one pass of the hot path over one synthetic batch (MNIST CNN: 32 samples per rank; ResNet-18: 64): forward
(bf16 autocast), backward, gradient all-reduce, optimizer, the step's tracked metrics and their cross-rank exchange —
EVERY step.  In the default (captured) mode the gradient all-reduce, the metric folds and the metric exchange are ONE
libdmlb kernel (fused step exchange) and the optimizer is one more (K5 / K6).  Everything goes through the public API:
TrainingPipeline.run() -> TrainValStage.train_epoch().

Timing.  Each arm below times exactly K = --steps steps, split into windows of at least 20 steps (one window when K < 40);
a window is one epoch with barrier + cuda synchronize around it, and CUDA events on the launching stream time its steps,
from handing out the first batch to the end of the last step (max over ranks).  One host hiccup can double a 5 ms window
(VERDICT r1), so value and e2e windows alternate and the MEDIAN time per step over the windows is reported (all window
times are in the JSON).  The number of steps the model trains for depends on the arguments only.

--dump-outputs DIR writes, after the timed steps, what the last step handed its caller (rank 0): the loss, the logits,
the parameters and buffers after the optimizer step, and the reduced train metrics of the last window, as DIR/<name>.npy
(float32; float64 for the buffers), at most 64 MB in all.  Such a run uses cuDNN's deterministic algorithms (as the MNIST
CNN always does) instead of autotuned ones, so that two runs with the same arguments compute the same outputs.

  value   inputs already resident in HBM (K distinct batches), device-timed, max over ranks
  e2e     the same loop fed from pinned HOST memory: H2D copy of every batch; the step's reduced metrics land in mapped
          host memory (written by the exchange kernel itself) and the host reads them, two steps late, every step
  roofline            libdmlb bucket kernel (dmlb_bucket_pack_f32_bf16) on a 1 GiB cold buffer, same C-ABI entry point
  roofline_in_situ    the gradient-sync launch on the real flat bucket of this workload
  cpu_baseline        the reference's CPU path on this box's host cores (rank 0, N=1 only): oracle/_ref (the installed,
                      unmodified reference) when present, else the restatement oracle/ref_port.py

Self-checks (exit non-zero): the peer communicator / CUDA graph silently unavailable at W > 1; e2e faster than value by
more than 2 %; replicas not bit-identical after the run; an oracle object injected into the product path.
Prints exactly one JSON line on rank 0.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))
# the tree may be read-only: no bytecode caches are written into it, by this process or the ones it spawns
sys.dont_write_bytecode = True
os.environ['PYTHONDONTWRITEBYTECODE'] = '1'

WORKLOADS = {
    'mnist': {'metric': 'samples/sec (box, device-timed) MNIST CNN', 'batch': 32, 'shape': (1, 28, 28), 'classes': 10,
              'name': 'MNIST CNN (examples/mnist.py:27-36) DDP, bf16 autocast, Adam, 32 samples/rank/step, 5 metrics '
                      'tracked + cross-rank metric exchange every step'},
    'resnet18': {'metric': 'samples/sec (box, device-timed) ResNet-18', 'batch': 64, 'shape': (3, 224, 224),
                 'classes': 1000,
                 'name': 'ResNet-18 (torchvision, 11,689,512 parameters) on synthetic 3x224x224 batches, DDP, bf16 '
                         'autocast, SGD momentum 0.9, 64 samples/rank/step, 5 metrics + cross-rank exchange every step'},
}
LABEL_BYTES = 8


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=100)
    ap.add_argument('--warmup', type=int, default=20)
    ap.add_argument('--impl', choices=['native', 'reference'], default='native')
    ap.add_argument('--workload', choices=sorted(WORKLOADS), default='mnist')
    ap.add_argument('--min-seconds', type=float, default=0.5,
                    help='reference arm: timed region (windows of K steps are repeated)')
    ap.add_argument('--grad-wire', choices=['bf16', 'fp32'], default='bf16')
    ap.add_argument('--grad-route', choices=['auto', 'peer', 'nccl'], default='auto')
    ap.add_argument('--grad-algo', type=int, default=0, help='dmlb_comm_allreduce algo: 0 auto, 1 one-shot, 2 two-shot, 3 NVLS')
    ap.add_argument('--metric-route', choices=['auto', 'peer', 'collective'], default='auto')
    ap.add_argument('--no-graph', action='store_true', help='eager step loop instead of the whole-step CUDA graph')
    ap.add_argument('--optim', choices=['flat', 'torch'], default='flat',
                    help='optimizer of the step: dmlcloud_b200.optim.FlatAdam / FlatSGD (libdmlb K5 / K6, one launch over '
                         'flat buffers, device-resident lr) or the torch optimizer (capturable)')
    ap.add_argument('--channels-last', choices=['auto', 'on', 'off'], default='auto',
                    help='keep model + images in NHWC, cuDNN\'s native bf16 layout.  auto = on for ResNet-18 (measured 2.05x: '
                         '12,316 vs 5,992 samples/s at N=1), off for the MNIST CNN (1-channel input; measured 5 %% slower)')
    ap.add_argument('--checkpoint-every-epoch', action='store_true',
                    help='BASELINE config 3: snapshot model/optimizer/tracker state after every window (= epoch)')
    ap.add_argument('--no-micro', action='store_true', help='skip the kernel / metric microbenchmarks')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR', help='native arm: write the last step\'s outputs as DIR/<name>.npy')
    args = ap.parse_args()
    args.channels_last = args.channels_last == 'on' or (args.channels_last == 'auto' and args.workload == 'resnet18')
    return args


# ----------------------------------------------------------------------------------------------------------------------
# clocks
# ----------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region (B200_PROFILING.md).  The region can be as short as
    0.1 s, so NVML is polled from a thread every 2 ms (an `nvidia-smi -lms` subprocess would not deliver a single sample
    in that time); nvidia-smi is only the fallback when the NVML bindings are missing."""
    REASONS = {'hw_slowdown': 0x8, 'hw_thermal_slowdown': 0x40, 'sw_thermal_slowdown': 0x20, 'sw_power_cap': 0x4}

    def __init__(self, gpu_index):
        self.gpu_index = gpu_index
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thread = None
        self._nvml = None

    def _physical_index(self):
        vis = os.environ.get('CUDA_VISIBLE_DEVICES')
        if vis:
            ids = [v.strip() for v in vis.split(',') if v.strip()]
            if self.gpu_index < len(ids) and ids[self.gpu_index].isdigit():
                return int(ids[self.gpu_index])
        return self.gpu_index

    def start(self):
        try:
            import pynvml

            pynvml.nvmlInit()
            self._nvml = pynvml
            self._handle = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index())
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self._handle, pynvml.NVML_CLOCK_SM))
        except Exception:  # noqa: BLE001
            self._nvml = None
            return
        self._poll()  # at least one sample even for a very short region
        self._thread = threading.Thread(target=self._run, daemon=True)
        self._thread.start()

    def _poll(self):
        nv = self._nvml
        try:
            self.samples.append(float(nv.nvmlDeviceGetClockInfo(self._handle, nv.NVML_CLOCK_SM)))
            mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self._handle)) if hasattr(
                nv, 'nvmlDeviceGetCurrentClocksEventReasons') else int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._handle))
            for name, bit in self.REASONS.items():
                if mask & bit:
                    self.reasons.add(name)
        except Exception:  # noqa: BLE001
            pass

    def _run(self):
        while not self._stop.wait(0.002):
            self._poll()

    def stop(self):
        if self._nvml is None:
            return self._smi_once()
        self._stop.set()
        if self._thread is not None:
            self._thread.join(timeout=2)
        self._poll()
        return {'sm_mhz': statistics.median(self.samples) if self.samples else None, 'sm_max_mhz': self.max_mhz,
                'samples': len(self.samples), 'reasons': sorted(self.reasons), 'how': 'NVML polled every 2 ms'}

    def _smi_once(self):
        try:
            out = subprocess.run(['nvidia-smi', '--query-gpu=clocks.sm,clocks.max.sm', '--format=csv,noheader,nounits',
                                  '-i', str(self._physical_index())], capture_output=True, text=True, timeout=10).stdout
            sm, mx = [float(v) for v in out.strip().split(',')[:2]]
            return {'sm_mhz': sm, 'sm_max_mhz': mx, 'samples': 1, 'reasons': [], 'how': 'nvidia-smi, once, after the region'}
        except Exception:  # noqa: BLE001
            return {'sm_mhz': None, 'sm_max_mhz': None, 'samples': 0, 'reasons': ['no NVML / nvidia-smi']}


# ----------------------------------------------------------------------------------------------------------------------
# native arm
# ----------------------------------------------------------------------------------------------------------------------
def native_arm(args):
    import contextlib
    import io
    import tempfile

    import torch
    import torch.distributed as dist
    from torch import nn

    from dmlcloud_b200 import TrainValStage, _native as N
    from dmlcloud_b200.metrics import DeviceSlab
    from dmlcloud_b200.pipeline import TrainingPipeline
    from dmlcloud_b200.util import distributed as D

    if not torch.cuda.is_available():
        raise SystemExit('bench.py (native arm) needs CUDA: dmlcloud_b200 has no CPU fallback')
    D.init_process_group_auto()
    world, rank = dist.get_world_size(), dist.get_rank()
    if world != args.gpus:
        raise SystemExit(f'--gpus {args.gpus} but WORLD_SIZE is {world}: launch with torchrun --nproc-per-node {args.gpus}')
    wl = WORKLOADS[args.workload]
    BATCH = wl['batch']
    use_graph = not args.no_graph
    eager_steps = 3 if args.workload == 'mnist' else 8  # (ResNet-18: the extra eager steps time DDP's rebuilt buckets)
    # graph mode spends the eager steps + 1 capture step before the first replay: keep all of that inside the warm-up
    K, W = args.steps, max(eager_steps + 5 if use_graph else 3, args.warmup)
    plan = window_plan(K)
    # cuDNN autotuning picks ResNet-18 convolutions 1.7 % faster than cuDNN's deterministic choice (B200, 1000 W).  On the
    # MNIST CNN the step it leads to took 0.236-0.252 ms in 8 of 10 processes, against 0.231-0.233 ms in every process
    # without it.  It may also pick other algorithms, hence other roundings, from run to run: runs whose outputs are
    # compared do without it.
    autotune = args.workload == 'resnet18' and not args.dump_outputs
    torch.backends.cudnn.benchmark = autotune
    torch.backends.cudnn.deterministic = not autotune

    def per_step(window_ms):
        return [ms / n for ms, n in zip(window_ms, plan)]

    def gen_batches(seed, count, pinned):
        g = torch.Generator().manual_seed(seed)
        out = []
        for _ in range(count):
            x = torch.randn(BATCH, *wl['shape'], generator=g)
            y = torch.randint(0, wl['classes'], (BATCH,), generator=g)
            out.append((x.pin_memory(), y.pin_memory()) if pinned else (x, y))
        return out

    def all_max(x):
        box = [None] * world
        dist.all_gather_object(box, x)
        return max(box)

    class BenchStage(TrainValStage):
        def pre_stage(self):
            dev = self.device
            torch.manual_seed(0)
            if args.workload == 'mnist':
                model = nn.Sequential(nn.Conv2d(1, 16, 3, padding=1), nn.ReLU(), nn.MaxPool2d(2),
                                      nn.Conv2d(16, 16, 3, padding=1), nn.ReLU(), nn.MaxPool2d(2), nn.Flatten(),
                                      nn.Linear(784, 10))  # reference examples/mnist.py:27-36
            else:
                import torchvision

                model = torchvision.models.resnet18()  # BASELINE config 4 (plain BatchNorm: sync_bn stays off)
            if args.channels_last:
                model = model.to(memory_format=torch.channels_last)
            self.pipeline.register_model('net', model, verbose=False, grad_wire=args.grad_wire)
            sync = self.pipeline.grad_syncs['net']
            sync.algo = args.grad_algo
            if args.optim == 'flat':  # libdmlb K5 / K6: parameters, state and (captured step) gradients in flat buffers
                from dmlcloud_b200.optim import FlatAdam, FlatSGD

                optimizer = (FlatAdam(model.parameters(), lr=1e-3) if args.workload == 'mnist'
                             else FlatSGD(model.parameters(), lr=0.1, momentum=0.9))
            elif args.workload == 'mnist':
                optimizer = torch.optim.Adam(model.parameters(), lr=1e-3, capturable=use_graph, fused=True)
            else:
                optimizer = torch.optim.SGD(model.parameters(), lr=0.1, momentum=0.9)
                for g in optimizer.param_groups:
                    g['capturable'] = True  # (SGD keeps no step tensor: it is capture-safe as it is)
            self.pipeline.register_optimizer('opt', optimizer)
            self.loss = nn.CrossEntropyLoss()
            # LOUD failure instead of silently timing another path (VERDICT r1): at W > 1 the bench needs the peer route
            if world > 1 and args.grad_route != 'nccl' and sync.comm is None:
                raise SystemExit('bench.py: the peer-memory communicator could not be created at W > 1 '
                                 '(pass --grad-route nccl --no-graph to time the NCCL route on purpose)')
            self.cuda_graph = use_graph
            self.cuda_graph_warmup = eager_steps
            self.live_metrics_every = 1  # metrics cross ranks EVERY step (BASELINE configs 2/3)
            self.manual_gc = True        # Python's cyclic GC runs at epoch boundaries, not inside a step (stage.py)
            self.tracker.deferred = True
            self.host = gen_batches(100 + rank, max(W, K), pinned=True)
            self.resident = [(x.to(dev), y.to(dev)) for x, y in self.host]
            self.pipeline.datasets['train'] = []
            self.pipeline.datasets['val'] = []
            self.windows = {'value': [], 'e2e': []}  # device ms per window (this rank)
            self.walls = {'value': [], 'e2e': []}
            self.launches = {'value': [], 'e2e': []}
            self.clocks = None
            self.host_reads = 0
            self.read_host = False
            self._older = None
            self.checkpoint_ms = []

        def step(self, batch):
            x, y = batch
            x = x.to(self.device, non_blocking=True)  # no-op for the resident phases
            if args.channels_last:
                x = x.contiguous(memory_format=torch.channels_last)
            y = y.to(self.device, non_blocking=True)
            with torch.autocast('cuda', dtype=torch.bfloat16):
                out = self.pipeline.models['net'](x)
            loss = self.loss(out.float(), y)
            self.track_reduce('accuracy', (out.argmax(1) == y).float().mean())
            # in a captured step these are the graph's static outputs: every replay rewrites them
            self.last_loss_logits = (loss.detach(), out.detach())
            return loss

        def table_columns(self):
            return [{'name': 'Epoch', 'metric': 'misc/epoch'}, {'name': 'Time/Epoch', 'metric': None},
                    {'name': 'Loss', 'metric': 'train/loss'}]

        def feed(self, data, events=None):
            """The 'DataLoader': hands out the next batch; in the e2e phase it first reads, on the host, the reduced
            metrics of two steps ago out of the mapped result ring (what a progress bar would print).  In a timed window
            `events` bracket the steps themselves: the first is recorded before the first batch is handed out, the second
            when the loop asks for a batch after the last step, so the epoch's set-up around them is not timed."""
            if events is not None:
                self.wall0 = time.perf_counter()
                events[0].record()
            for batch in data:
                if self.read_host:
                    if self._older is not None and 'train/loss' in self._older:
                        self.last_loss = self._older['train/loss'].value()
                        self.host_reads += 1
                    self._older = self.live_metrics or None
                yield batch
            if events is not None:
                events[1].record()

        def _window(self, kind):
            i = len(self.windows[kind])
            start = sum(plan[:i])
            data = (self.resident if kind == 'value' else self.host)[start:start + plan[i]]
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            self.pipeline.datasets['train'] = self.feed(data, (t0, t1))
            self.read_host, self._older = kind == 'e2e', None
            # the polling thread takes the GIL from the host-bound step loop: it runs beside the first e2e window, not
            # beside the headline arm (whose first window is its only one when K < 40)
            sampler = ClockSampler(self.device.index) if (kind == 'e2e' and self.clocks is None) else None
            dist.barrier()
            torch.cuda.synchronize()
            if sampler:
                sampler.start()
            n0 = N.launch_count()
            replays0 = self._graph.replays if self._graph is not None else 0
            self.train_epoch()  # <- the public per-step loop (stage.py train_epoch) over this window's steps
            torch.cuda.synchronize()
            wall = (time.perf_counter() - self.wall0) * 1e3
            dist.barrier()
            if sampler:
                self.clocks = sampler.stop()
            launches = N.launch_count() - n0  # launched through the C ABI in the region ...
            if self._graph is not None:        # ... plus the libdmlb kernels each graph replay re-runs
                launches += (self._graph.replays - replays0) * self._graph.kernels_in_graph
            self.windows[kind].append(max(t0.elapsed_time(t1), 0.0))
            self.walls[kind].append(wall)
            self.launches[kind].append(launches)

        def run_epoch(self):
            e = self.current_epoch
            if e == 1:  # warm-up on resident data: eager steps, capture, first replays (also cuDNN autotuning)
                sync = self.pipeline.grad_syncs['net']
                sync.profile_events = args.workload != 'mnist'  # DDP's (rebuilt) buckets through the hook, timed in situ
                self.pipeline.datasets['train'] = self.feed(self.resident[:W])
                self.train_epoch()
                sync.profile_events = False
                return
            if e == 2:  # warm-up of the host-fed loop
                self.pipeline.datasets['train'] = self.feed(self.host[:min(W, 8)])
                self.read_host = True
                self.train_epoch()
                if use_graph and self._graph is None:
                    raise SystemExit('bench.py: the whole-step CUDA graph was not captured during the warm-up')
                return
            self._window('value' if e % 2 == 1 else 'e2e')  # windows alternate so that drift hits both arms alike
            if len(self.windows['e2e']) == len(plan):
                v = statistics.median(per_step(self.windows['value']))
                x = statistics.median(per_step(self.windows['e2e']))
                # e2e does strictly more work than value: if it measures faster by > 2 % the windows were too noisy
                self.inconsistent = bool(all_max(1 if x < 0.98 * v else 0))
                self.stop_stage()

        def post_epoch(self):
            if args.checkpoint_every_epoch and self.pipeline.last_checkpoint_ms is not None:
                self.checkpoint_ms.append(self.pipeline.last_checkpoint_ms)

    pipeline = TrainingPipeline(name='bench')
    pipeline.grad_route, pipeline.metric_route = args.grad_route, args.metric_route
    if args.checkpoint_every_epoch:
        root = [tempfile.mkdtemp(prefix='dmlb_bench_ckpt_') if rank == 0 else None]
        dist.broadcast_object_list(root, src=0)
        pipeline.enable_checkpointing(root[0])
    stage = BenchStage()
    pipeline.append_stage(stage, max_epochs=None)
    with contextlib.redirect_stdout(io.StringIO()):
        pipeline.run()
    dev = pipeline.device
    sync = pipeline.grad_syncs['net']
    graph = stage._graph

    # ---- honesty checks -------------------------------------------------------------------------------------------------
    if not isinstance(pipeline.tracker._slab, DeviceSlab):
        raise SystemExit('bench.py: the metric slab is not the CUDA slab (a test seam leaked into the product path)')
    if getattr(pipeline.optimizers['opt'], '_lib_override', None) is not None:
        raise SystemExit('bench.py: the optimizer runs on an injected library, not libdmlb')
    if use_graph and graph is None:
        raise SystemExit('bench.py: the whole-step CUDA graph is not active')
    if getattr(stage, 'inconsistent', False):
        raise SystemExit(f'bench.py: e2e measured faster than value by more than 2 % after {len(stage.windows["value"])} '
                         f'windows per arm: value {statistics.median(stage.windows["value"]):.4f} ms, '
                         f'e2e {statistics.median(stage.windows["e2e"]):.4f} ms per window')
    # replicas must be bit-identical after thousands of steps over the real NVLink peers (driver-visible correctness)
    with torch.no_grad():
        flat = torch.cat([p.detach().flatten() for p in pipeline.models['net'].parameters()])
        digest = (int(flat.view(torch.int32).to(torch.int64).sum().item()), float(flat.double().sum().item()))
    digests = [None] * world
    dist.all_gather_object(digests, digest)
    replicas_identical = all(d == digests[0] for d in digests)
    if not replicas_identical:
        raise SystemExit(f'bench.py: model replicas diverged across ranks: {digests}')
    if not all(torch.isfinite(flat.double().sum()).item() for _ in (0,)):
        raise SystemExit('bench.py: non-finite parameters after the run')
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, stage, pipeline)

    # ---- numbers ---------------------------------------------------------------------------------------------------------
    def gathered_windows(kind):
        """max over ranks, window by window (every rank timed the same windows)"""
        box = [None] * world
        dist.all_gather_object(box, stage.windows[kind])
        return [max(col) for col in zip(*box)]

    value_windows, e2e_windows = gathered_windows('value'), gathered_windows('e2e')
    box = [None] * world
    dist.all_gather_object(box, stage.walls['e2e'])
    e2e_walls = [max(col) for col in zip(*box)]
    step_ms = statistics.median(per_step(value_windows))
    # host reads are part of e2e: per window the larger of the device time and the host wall time
    e2e_step_ms = statistics.median(per_step([max(d, w) for d, w in zip(e2e_windows, e2e_walls)]))
    samples = BATCH * world  # per step

    # ---- in-situ gradient sync timing ----
    torch.cuda.synchronize()
    peaks = load_peaks()
    in_situ, buckets_in_situ = None, []
    if graph is not None:  # inside the graph no event can be recorded: time the same launch right after
        durs = graph.time_gradient_sync()[3:]
        n_elem = graph.bucket.total
        route = 'single' if world == 1 else 'peer'
        wire_b = 2 if args.grad_wire == 'bf16' else 4
        mean_us = statistics.mean(durs)
        if world == 1:  # read fp32 + write fp32 in place (rounded through the wire dtype in registers)
            alg = n_elem * 8
            in_situ = {'kernel': f'dmlb_comm_allreduce[W=1,{args.grad_wire}] on the flat gradient bucket', 'bound': 'hbm',
                       'achieved': round(alg / (mean_us * 1e-6) / 1e9, 2), 'peak': peaks['hbm_gbs'], 'unit': 'GB/s'}
        else:  # bus bandwidth convention: 2 (W-1)/W x wire bytes over the NVLink time
            alg = int(2 * (world - 1) / world * n_elem * wire_b)
            in_situ = {'kernel': f'dmlb_comm_allreduce[W={world},{args.grad_wire}] on the flat gradient bucket',
                       'bound': 'nvlink', 'achieved': round(alg / (mean_us * 1e-6) / 1e9, 2), 'peak': NVLINK_GBPS,
                       'unit': 'GB/s (bus bandwidth)'}
        in_situ.update({'elements': n_elem, 'frac': round(in_situ['achieved'] / in_situ['peak'], 5),
                        'mean_us': round(mean_us, 2), 'algorithmic_bytes_per_launch': alg, 'launches_timed': len(durs),
                        'note': 'the bucket is L2-resident right after backward; MNIST (41 KB) is launch-latency bound'})
    if sync.event_log:  # DDP's own buckets through the hook during the eager warm-up steps (ResNet-18: 3 rebuilt buckets)
        per = {}
        for a, b, n, r in sync.event_log:
            per.setdefault((n, r), []).append(a.elapsed_time(b) * 1e3)
        for (n, r), us in sorted(per.items()):
            us = statistics.median(us)
            wire_b = 2 if args.grad_wire == 'bf16' else 4
            e = {'elements': n, 'route': r, 'median_us': round(us, 2), 'launches_timed': len(per[(n, r)])}
            if world > 1:
                e['bus_GBps'] = round(2 * (world - 1) / world * n * wire_b / (us * 1e-6) / 1e9, 1)
                e['frac_of_nvlink'] = round(e['bus_GBps'] / NVLINK_GBPS, 3)
            else:
                e['hbm_GBps'] = round(n * 8 / (us * 1e-6) / 1e9, 1)
                e['frac_of_hbm'] = round(e['hbm_GBps'] / peaks['hbm_gbs'], 3)
            buckets_in_situ.append(e)

    live_cells = sum(m.lanes for m in graph.live_names.values()) if graph is not None and graph.live_names else \
        sum(m.lanes for m in pipeline.tracker.live_selection()[0].values())
    result = {
        'metric': wl['metric'], 'value': round(samples / (step_ms * 1e-3), 1), 'unit': 'samples/s', 'n_gpus': world,
        'steps': K, 'warmup': W, 'ms_per_step': round(step_ms, 4), 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'bf16' if args.grad_wire == 'bf16' else 'f32', 'data': 'synthetic',
        'config': {'workload': wl['name'], 'global_batch': BATCH * world, 'parallelism': f'dp{world}',
                   'grad_wire': args.grad_wire, 'cuda_graph': bool(graph is not None),
                   'channels_last': bool(args.channels_last),
                   'optimizer': type(pipeline.optimizers['opt']).__name__,
                   'graph_replays': graph.replays if graph is not None else 0,
                   'kernels_per_step': graph.kernels_in_graph if graph is not None else None,
                   'step_exchange': 'fused into the gradient all-reduce kernel (one launch per step; LL protocol — data and flag pushed together, no separate barrier — for messages <= 256 KB)'
                   if graph is not None and graph.step_metrics is not None else 'separate exchange kernel',
                   'grad_route': sorted(set(sync.last_routes.values())) if graph is None else
                   ['single' if world == 1 else 'peer'],
                   'multicast': bool(sync.comm is not None and sync.comm.multicast),
                   'python_gc': 'cyclic collector runs at epoch (= window) boundaries, not inside the step loop (stage.manual_gc)',
                   'metric_route': 'peer' if (pipeline.metric_comm is not None or graph is not None) else
                   ('single' if world == 1 else 'collective'),
                   'timing': f'{K} steps per arm in windows of {plan} steps (value / e2e alternating), median time per '
                             'step over the windows; each window bracketed by barrier + synchronize, CUDA events, max '
                             'over ranks',
                   'l2': ('K distinct batches; the MNIST working set (<10 MB) is L2-resident by the nature of the workload'
                          if args.workload == 'mnist' else
                          'K distinct batches of 38.5 MB each + 45 MB of gradients per step: larger than the 126 MB L2') +
                         '; the roofline microbench uses 1 GiB buffers'},
        'clocks': stage.clocks,
        'e2e': {'value': round(samples / (e2e_step_ms * 1e-3), 1), 'unit': 'samples/s',
                'h2d_bytes_per_step': BATCH * (4 * wl['shape'][0] * wl['shape'][1] * wl['shape'][2] + LABEL_BYTES),
                'd2h_bytes_per_step': 12 + 9 * live_cells,  # stamp + status + {value, flag} per exchanged cell, written
                'ms_per_step': round(e2e_step_ms, 4), 'host_reads': stage.host_reads,   # into mapped host memory
                'windows_ms': [round(w, 3) for w in e2e_windows]},
        'gpu_launches': int(statistics.median(stage.launches['value'])),
        'windows_ms': [round(w, 3) for w in value_windows],
        'window_steps': plan,
        'window_spread': {'min_ms': round(min(value_windows), 3), 'max_ms': round(max(value_windows), 3)},
        'wall_ms_per_step': round(statistics.median(per_step(stage.walls['value'])), 4),
        'replicas_identical': replicas_identical,
        'roofline_in_situ': in_situ,
    }
    if buckets_in_situ:
        result['ddp_buckets_in_situ'] = buckets_in_situ
    if args.checkpoint_every_epoch:
        ms = stage.checkpoint_ms
        result['checkpoint'] = {'every': 'window (= one epoch)', 'snapshots': len(ms),
                                'host_ms_per_epoch_median': round(statistics.median(ms), 3) if ms else None,
                                'host_ms_per_epoch_max': round(max(ms), 3) if ms else None,
                                'what': 'wall time the epoch loop spends on the snapshot (D2H into pinned staging is '
                                        'queued on a side stream; rank 0 writes the file on a background thread)'}

    if rank == 0 and not args.no_micro:
        result.update(kernel_microbench(dev, peaks))
    if not args.no_micro:
        mr = metric_reduce_microbench(pipeline, dev, world, rank)
        if rank == 0:
            result['metric_reduce_us'] = mr
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        result['cpu_baseline'] = cpu_baseline(args)
    dist.barrier()
    if rank == 0:
        print(json.dumps(result), file=JSON_OUT, flush=True)
    pipeline.wait_for_checkpoints()
    for s_ in pipeline.grad_syncs.values():
        s_.close()
    if pipeline.metric_comm is not None:
        pipeline.metric_comm.close()
    dist.destroy_process_group()


def window_plan(k, min_steps=20):
    """k timed steps as windows of at least `min_steps` steps each (one window when k < 2 * min_steps)."""
    n = max(1, k // min_steps)
    return [k // n + (i < k % n) for i in range(n)]


DUMP_BYTES = 64 << 20


def dump_outputs(directory, stage, pipeline):
    """What the last timed step handed its caller, as <directory>/<name>.npy: its loss and logits, the model's
    parameters and buffers after the optimizer step, and the train metrics reduced over the last window."""
    import numpy as np
    import torch

    torch.cuda.synchronize()
    model = pipeline.models['net']
    loss, logits = stage.last_loss_logits
    with torch.no_grad():
        arrays = {'loss': loss.float().cpu().numpy(), 'logits': logits.float().cpu().numpy(),
                  'parameters': torch.cat([p.flatten().float() for p in model.parameters()]).cpu().numpy()}
        buffers = [b.flatten().double() for b in model.buffers()]
        if buffers:
            arrays['buffers'] = torch.cat(buffers).cpu().numpy()
        for name in ('train/loss', 'train/accuracy'):
            arrays[name.replace('/', '_')] = torch.as_tensor(pipeline.tracker[name][-1]).float().cpu().numpy()
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_BYTES:
        raise SystemExit(f'bench.py: the outputs take {total} bytes, more than --dump-outputs writes ({DUMP_BYTES})')
    out = Path(directory)
    out.mkdir(parents=True, exist_ok=True)
    for name, a in arrays.items():
        np.save(out / f'{name}.npy', a)


NVLINK_GBPS = 770.0  # measured per-direction peer bandwidth of this pool's B200s (B200_PROFILING.md; spec 900)


def load_peaks():
    p = ROOT / 'MEASURED_PEAKS.json'
    if p.exists():
        d = json.loads(p.read_text())
        return {'hbm_gbs': float(d['hbm_gbs']), 'source': 'MEASURED_PEAKS.json (of measured)'}
    return {'hbm_gbs': 6650.0, 'source': 'B200_PROFILING.md fallback (of fallback)'}


def ncu_traffic(kernel_substr):
    """DRAM bytes (read + write) per launch of a kernel from the committed `ncu --set full` summary of the same 1 GiB
    launch (profiles/r2_bucket_kernels_ncu_full.csv, made by profiles/summarize_ncu.py); None if absent."""
    import csv

    path = ROOT / 'profiles' / 'r2_bucket_kernels_ncu_full.csv'
    if not path.exists():
        return None
    rows = list(csv.reader(open(path)))
    head = rows[0]
    try:
        k, t = head.index('Kernel Name'), head.index('dram_bytes_total')
    except ValueError:
        return None
    for r in rows[2:]:
        if kernel_substr in r[k]:
            return int(float(r[t]))
    return None


def kernel_microbench(dev, peaks):
    """The bucket kernels through the C ABI on buffers far larger than L2 (1 GiB fp32 source), CUDA-event timed per launch
    on the launching stream; plus the ResNet-18 bucket sizes with an L2 flush between launches."""
    import torch

    from dmlcloud_b200 import _native as N

    lib = N.cuda_lib(dev.index)
    n = 1 << 28  # 268,435,456 fp32 = 1 GiB
    src = torch.empty(n, dtype=torch.float32, device=dev).normal_()
    wire = torch.empty(n, dtype=torch.bfloat16, device=dev)
    st = N.stream_ptr()

    def timed(fn, reps=10, warm=3, between=None):
        for _ in range(warm):
            fn()
        out = []
        for _ in range(reps):
            if between:
                between()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            b.synchronize()
            out.append(a.elapsed_time(b) * 1e-3)
        return out

    def entry(name, bytes_per_elem, elems, secs, note=None):
        mean = statistics.mean(secs)
        ach = elems * bytes_per_elem / mean / 1e9
        d = {'kernel': name, 'bound': 'hbm', 'achieved': round(ach, 1), 'peak': peaks['hbm_gbs'], 'unit': 'GB/s',
             'frac': round(ach / peaks['hbm_gbs'], 4), 'traffic': None, 'elements': elems,
             'algorithmic_bytes_per_launch': elems * bytes_per_elem, 'mean_us': round(mean * 1e6, 2),
             'best_us': round(min(secs) * 1e6, 2), 'peak_source': peaks['source']}
        if note:
            d['note'] = note
        return d

    pack = timed(lambda: N.check(lib.dmlb_bucket_pack_f32_bf16(src.data_ptr(), wire.data_ptr(), n, 0.125, st)))
    pack_tma = timed(lambda: N.check(lib.dmlb_bucket_pack_f32_bf16_tma(src.data_ptr(), wire.data_ptr(), n, 0.125, st)))
    pack_regs = timed(lambda: N.check(lib.dmlb_bucket_pack_f32_bf16_regs(src.data_ptr(), wire.data_ptr(), n, 0.125, st)))
    unpack_tma = timed(lambda: N.check(lib.dmlb_bucket_unpack_bf16_f32_tma(wire.data_ptr(), src.data_ptr(), n, 1.0, st)))
    unpack_regs = timed(lambda: N.check(lib.dmlb_bucket_unpack_bf16_f32_regs(wire.data_ptr(), src.data_ptr(), n, 1.0,
                                                                             None, st)))
    unpack = timed(lambda: N.check(lib.dmlb_bucket_unpack_bf16_f32(wire.data_ptr(), src.data_ptr(), n, 1.0, None, st)))
    scale = timed(lambda: N.check(lib.dmlb_bucket_scale_f32(src.data_ptr(), n, 1.0, st)))
    sq = torch.zeros(1, dtype=torch.float64, device=dev)
    read_only = timed(lambda: N.check(lib.dmlb_bucket_sumsq_f32(src.data_ptr(), n, sq.data_ptr(), st)))
    write_only = timed(lambda: src.zero_())  # cudaMemset-class fill by torch: context for the write-heavy kernels
    q = n // 4  # K5 on four quarter-size arrays carved out of `src` (all zero after the fill above: timing only)
    adam_state = torch.zeros(2, dtype=torch.int64, device=dev)
    quarters = [src.data_ptr() + 4 * q * i for i in range(4)]
    adam = timed(lambda: N.check(lib.dmlb_adam_step_f32(quarters[0], quarters[1], quarters[2], quarters[3], q, 1e-3, 0.9,
                                                        0.999, 1e-8, 0.0, 0, 0, None, 0.0, adam_state.data_ptr(), 1, None,
                                                        0, st)))
    traffic = {'pack': ncu_traffic('pack_bf16_tma_kernel'), 'pack_regs': ncu_traffic('PackBf16'),
               'unpack_tma': ncu_traffic('unpack_bf16_tma_kernel'), 'unpack_regs': ncu_traffic('UnpackBf16'),
               'scale': ncu_traffic('ScaleInplace')}
    out = {
        'hbm_context': {'read_only_GBps': round(n * 4 / statistics.mean(read_only) / 1e9, 1),
                        'write_only_GBps': round(n * 4 / statistics.mean(write_only) / 1e9, 1),
                        'note': 'read-only = dmlb_bucket_sumsq_f32 (4 B/el); write-only = torch zero_ fill (4 B/el); '
                                'the measured copy peak is a 50/50 read/write mix'},
        'roofline': entry('dmlb_bucket_pack_f32_bf16 (K1, default dispatch)', 6, n, pack,
                          'microbench through the same C-ABI entry point on a 1 GiB fp32 source (cold: > 126 MB L2); '
                          'traffic = dram__bytes_read.sum + dram__bytes_write.sum of the same launch from the committed '
                          'ncu --set full capture (profiles/r2_bucket_kernels_ncu_full.csv)'),
        'roofline_more': [entry('dmlb_bucket_pack_f32_bf16_tma (K1 via TMA bulk loads)', 6, n, pack_tma),
                          entry('dmlb_bucket_pack_f32_bf16_regs (K1 via LDG.128 x4 in registers)', 6, n, pack_regs),
                          entry('dmlb_bucket_unpack_bf16_f32 (K2, default dispatch)', 6, n, unpack),
                          entry('dmlb_bucket_unpack_bf16_f32_tma (K2 via TMA bulk load + bulk store)', 6, n, unpack_tma),
                          entry('dmlb_bucket_unpack_bf16_f32_regs (K2 via registers)', 6, n, unpack_regs),
                          entry('dmlb_bucket_scale_f32 (K1, fp32 wire, in place)', 8, n, scale),
                          entry('dmlb_adam_step_f32 (K5, Adam step on a flat bucket: 16 B read + 12 B written per element)',
                                28, q, adam)],
    }
    # ResNet-18 DDP buckets (SURVEY §8a-3).  A single 10 us launch cannot be timed with an event pair (the pair itself
    # costs microseconds), so R x [L2 flush, kernel] is captured into a CUDA graph and timed against R x [L2 flush].
    flush = torch.empty(64 << 20, dtype=torch.float32, device=dev)  # 256 MB write > 126 MB L2
    side = torch.cuda.Stream(device=dev)

    def graph_time(body, reps=8, R=8):
        g = torch.cuda.CUDAGraph()
        with torch.cuda.stream(side):
            body()
            torch.cuda.synchronize()
            with torch.cuda.graph(g, stream=side):
                for _ in range(R):
                    body()
            ts = []
            for _ in range(reps):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                g.replay()
                b.record()
                b.synchronize()
                ts.append(a.elapsed_time(b) * 1e-3 / R)
        return ts

    def side_ptr():
        return N.stream_ptr(torch.cuda.current_stream(dev))

    base = statistics.median(graph_time(lambda: flush.zero_()))

    def tiny():
        flush.zero_()
        N.check(lib.dmlb_bucket_scale_f32(src.data_ptr(), 4, 1.0, side_ptr()))

    # what ANY kernel node costs in this measurement (node-to-node launch gap + an empty grid's ramp): the floor under the
    # small buckets.  A 513,000-element bucket moves 3 MB = 0.47 us at the HBM peak; no stand-alone launch can take that
    # little, which is why the product path fuses the pack into the all-reduce kernel instead of launching it.
    floor_us = max(statistics.median(graph_time(tiny)) - base, 0.0) * 1e6
    out['launch_floor_us'] = round(floor_us, 2)
    buckets = []
    for elems in (513_000, 7_213_056, 3_963_456, 11_689_512):
        s = src[:elems]
        w = wire[:elems]

        def body():
            flush.zero_()
            N.check(lib.dmlb_bucket_pack_f32_bf16(s.data_ptr(), w.data_ptr(), elems, 0.125, side_ptr()))

        secs = [max(t - base, 1e-9) for t in graph_time(body)]
        buckets.append(entry('dmlb_bucket_pack_f32_bf16 (K1)', 6, elems, secs,
                             'cold: 256 MB L2 flush before each launch; graph-captured, flush time subtracted'))
        net = max(statistics.mean(secs) * 1e6 - floor_us, 1e-3)
        buckets[-1]['net_of_launch_floor_us'] = round(net, 2)
        buckets[-1]['frac_net_of_launch_floor'] = round(elems * 6 / (net * 1e-6) / 1e9 / peaks['hbm_gbs'], 4)
        for label, fn in (('regs', lib.dmlb_bucket_pack_f32_bf16_regs), ('tma', lib.dmlb_bucket_pack_f32_bf16_tma)):
            def body_v(fn=fn):
                flush.zero_()
                N.check(fn(s.data_ptr(), w.data_ptr(), elems, 0.125, side_ptr()))

            secs_v = [max(t - base, 1e-9) for t in graph_time(body_v)]
            buckets.append(entry(f'dmlb_bucket_pack_f32_bf16_{label}', 6, elems, secs_v, f'cold, {label} path forced'))
        # the same bucket as the step sees it: just written by backward, i.e. L2-resident
        warm = graph_time(lambda: N.check(lib.dmlb_bucket_pack_f32_bf16(s.data_ptr(), w.data_ptr(), elems, 0.125,
                                                                         side_ptr())))
        buckets.append(entry('dmlb_bucket_pack_f32_bf16 (K1)', 6, elems, warm,
                             'warm: source L2-resident (as right after backward); back-to-back in a graph'))
    out['roofline_resnet18_buckets'] = buckets
    out['roofline']['traffic'] = traffic['pack']
    for e in out['roofline_more']:
        for key, sub in (('pack_regs', '_regs (K1'), ('pack', '_tma (K1'), ('unpack_tma', 'f32_tma'), ('unpack_regs', 'f32_regs'),
                         ('scale', 'scale_f32')):
            if sub in e['kernel']:
                e['traffic'] = traffic[key]
    del src, wire, flush
    torch.cuda.empty_cache()
    return out


def metric_reduce_microbench(pipeline, dev, world, rank, n_metrics=1024):
    """BASELINE config 5: 1024 scalar metrics reduced per step.  Per step every metric gets a value, then the cross-rank
    exchange `reduce_live()` runs — ONE fused kernel (finalise + peer exchange + combine) writing straight into mapped
    pinned host memory — and the host reads a result.  Three variants:
      floats_mixed   python floats (kernel immediates), 256 each MEAN / SUM / MIN / MAX            (r1's variant)
      device_mean    0-d fp32 DEVICE tensors (torch.randn on the device, seed = rank), all MEAN    (BASELINE's wording)
      device_mixed   device tensors: 256 each MEAN / SUM / MIN / MAX fp32 + 64 int64 SUM counters
    Reported per variant (us, max over ranks): CUDA-event time of the call issued right after a host barrier (includes the
    ranks' launch skew), back-to-back (steady state of a step loop), device-aligned (queued behind a peer-barrier kernel:
    no host skew), host wall time of the call, and the epoch-closing next_epoch() incl. its host bookkeeping."""
    import torch
    import torch.distributed as dist

    from dmlcloud_b200.metrics import MetricTracker, Reduction

    ops = [Reduction.MEAN, Reduction.SUM, Reduction.MIN, Reduction.MAX]

    def stats(xs):
        xs = sorted(xs)
        return {'median': xs[len(xs) // 2], 'p99': xs[max(0, int(len(xs) * 0.99) - 1)], 'min': xs[0]}

    def variant(kind, iters, warm, gc_off=False):
        import gc

        if gc_off:
            gc.collect()
            gc.disable()
        t = MetricTracker()
        t.bind(device=dev, comm=pipeline.metric_comm, group=None)
        t.deferred = True
        names = [f'm{i}' for i in range(n_metrics)]
        for i, name in enumerate(names):
            t.register_metric(name, Reduction.MEAN if kind == 'device_mean' else ops[i % 4])
        counters = [f'c{i}' for i in range(64)] if kind == 'device_mixed' else []
        for name in counters:
            t.register_metric(name, Reduction.SUM)
        g = torch.Generator(device=dev).manual_seed(rank)
        if kind == 'floats_mixed':
            vals = torch.randn(n_metrics, generator=torch.Generator().manual_seed(rank)).tolist()
            cvals = []
        else:
            block = torch.randn(n_metrics, generator=g, device=dev)
            vals = list(block.unbind(0))  # 1024 separate 0-d device tensors (views of one block)
            cvals = list(torch.randint(0, 1000, (len(counters),), generator=g, device=dev).unbind(0))
        live_us, live_host_us, epoch_us, pipe_us, dev_us, parts = [], [], [], [], [], []
        for it in range(warm + iters):
            for name, v in zip(names, vals):
                t.track(name, v)
            for name, v in zip(counters, cvals):
                t.track(name, v)
            t._slab.flush_all()
            dist.barrier()
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            h0 = time.perf_counter()
            a.record()
            ha = time.perf_counter()
            live = t.reduce_live()
            hb = time.perf_counter()
            b.record()
            h1 = time.perf_counter()
            b.synchronize()
            assert live['m1'].value() is not None  # the host consumes every exchange's result (ring slots recycle)
            if it >= warm:
                live_us.append(a.elapsed_time(b) * 1e3)
                live_host_us.append((h1 - h0) * 1e6)
                parts.append(((ha - h0) * 1e6, (hb - ha) * 1e6, (h1 - hb) * 1e6))
            if it % 10 == 9:
                R = 10
                p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                p0.record()
                for _ in range(R):
                    keep = t.reduce_live()
                p1.record()
                p1.synchronize()
                keep['m1'].value()
                if it >= warm:
                    pipe_us.append(p0.elapsed_time(p1) * 1e3 / R)
                if pipeline.metric_comm is not None:
                    d0, d1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    pipeline.metric_comm.barrier()
                    d0.record()
                    keep = t.reduce_live()
                    d1.record()
                    d1.synchronize()
                    if it >= warm:
                        dev_us.append(d0.elapsed_time(d1) * 1e3)
                a2, b2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a2.record()
                t.next_epoch()
                b2.record()
                b2.synchronize()
                epoch_us.append(a2.elapsed_time(b2) * 1e3)
        t._materialize()
        mine = {'live': stats(live_us), 'host': stats(live_host_us), 'epoch': stats(epoch_us), 'pipe': stats(pipe_us),
                'dev': stats(dev_us) if dev_us else stats(pipe_us)}
        box = [None] * world
        dist.all_gather_object(box, mine)

        def worst(k):
            return {s_: round(max(b_[k][s_] for b_ in box), 2) for s_ in ('median', 'p99', 'min')}

        if gc_off:
            gc.enable()
        out = {'iters': iters}
        # where a slow call spends its HOST time (this rank): the timing event's record, the reduce_live() call, the end event
        slow = max(range(len(parts)), key=lambda i: sum(parts[i]))
        out['slowest_call_host_us'] = {'event_record_start': round(parts[slow][0], 1), 'reduce_live': round(parts[slow][1], 1),
                                       'event_record_end': round(parts[slow][2], 1)}
        out.update(worst('live'))
        out.update({'host_call': worst('host'), 'back_to_back': worst('pipe'), 'device_aligned': worst('dev'),
                    'next_epoch': worst('epoch')})
        return out

    out = {'n_metrics': n_metrics, 'world': world, 'unit': 'us'}
    out.update(variant('floats_mixed', 200, 20))  # top-level keys keep r1's meaning (python floats, mixed ops)
    # the p99 of the call-after-a-host-barrier numbers is a HOST stall between the start event and the launch; with the
    # Python garbage collector off during the loop it shows whether that stall is a gen-1/2 collection
    out['floats_mixed_gc_disabled'] = variant('floats_mixed', 200, 20, gc_off=True)
    out['device_mean'] = variant('device_mean', 60, 10)
    out['device_mixed_int64'] = variant('device_mixed', 60, 10)
    out['what'] = ('median/p99/min: CUDA-event time of MetricTracker.reduce_live() (fused reduce kernel writing into mapped '
                   'pinned host memory) with all metrics holding a value, issued right after a host barrier (includes the '
                   'ranks\' launch skew); back_to_back: per call when 10 exchanges are issued back to back; device_aligned '
                   '(W>1): one exchange queued behind a peer-barrier kernel, i.e. without host launch skew; host_call: wall '
                   'time of the Python call; next_epoch: CUDA-event time of the epoch-closing reduce incl. its O(#metrics) '
                   'host bookkeeping.  device_mean / device_mixed_int64: the same with 0-d DEVICE tensors as values')
    return out


def _run_reference(world, steps, warmup, workload, min_seconds):
    """The reference's CPU path on this box's host cores: the installed, unmodified reference (oracle/_ref) when it
    travelled with the snapshot, else the restatement (oracle/ref_port.py, MNIST only)."""
    from oracle import ref_port, ref_run

    if ref_run.available():
        try:
            return ref_run.run_baseline(world=world, steps=steps, warmup=warmup, total_threads=ref_run.usable_cores(),
                                        min_seconds=min_seconds, workload=workload)
        except Exception as exc:  # noqa: BLE001 - the installed reference failed to run on this box: say so, time the port
            print(f'bench.py: oracle/_ref could not be run ({type(exc).__name__}: {exc}); falling back to oracle/ref_port.py',
                  file=sys.stderr)
    if workload != 'mnist':
        raise SystemExit('bench.py: oracle/_ref (the installed reference) is needed for the ResNet-18 reference arm')
    cores = ref_port.usable_cores()
    stock = ref_port.run_baseline(world=world, steps=steps, warmup=max(3, warmup), total_threads=cores,
                                  per_step_reduce=False)
    strict = ref_port.run_baseline(world=world, steps=steps, warmup=max(3, warmup), total_threads=cores,
                                   per_step_reduce=True)
    stock.update({'kind': 'port', 'windows': 1, 'per_step_reduce_samples_per_s': strict['samples_per_s']})
    return stock


def _describe_reference(res, workload):
    batch = WORKLOADS[workload]['batch']
    what = ('the installed, unmodified reference (oracle/_ref: pip install --target of /root/reference) — its own '
            'TrainValStage + DDP over gloo on CPU tensors') if res['kind'] == 'reference' else \
        'oracle/ref_port.py, a restatement of the reference\'s CPU path (oracle/_ref did not travel)'
    return {'value': round(res['samples_per_s'], 1), 'unit': 'samples/s', 'cores': res['cores'], 'kind': res['kind'],
            'sample': f'median of {res.get("windows", 1)} windows of {res["steps"]} training steps x {batch} samples x '
                      f'{res["world"]} rank(s), {res["seconds"]:.1f} s of {what}; stock behaviour: metrics cross ranks once '
                      'per epoch (reference stage.py:180-185)',
            'threads_per_rank': res['threads_per_rank'], 'thread_calibration': res.get('calibration'),
            'epoch_reduce_ms': round(res['epoch_reduce_ms'], 3),
            'per_step_reduce_value': round(res['per_step_reduce_samples_per_s'], 1),
            'per_step_reduce_note': 'the same reference with tracker.next_epoch() after EVERY step — the operating point '
                                    'the native arm runs at (BASELINE configs 2/3); reported beside the stock number'}


def cpu_baseline(args):
    """N=1 leg: the reference's CPU path, W=1, bounded sample (>= 2 s of timed windows)."""
    res = _run_reference(1, min(args.steps, 50) if args.workload == 'mnist' else 2, 5, args.workload, 2.0)
    return _describe_reference(res, args.workload)


# ----------------------------------------------------------------------------------------------------------------------
# reference arm
# ----------------------------------------------------------------------------------------------------------------------
def reference_arm(args):
    """The reference's own CPU implementation of the path on this box's host cores, W = --gpus gloo ranks, as many host
    threads as help (calibrated once, on >= 48-step samples).  Under torchrun only rank 0 works."""
    if int(os.environ.get('RANK', '0')) != 0:
        return
    for k in ('RANK', 'WORLD_SIZE', 'LOCAL_RANK', 'MASTER_PORT', 'MASTER_ADDR', 'LOCAL_WORLD_SIZE', 'GROUP_RANK'):
        os.environ.pop(k, None)  # the baseline spawns its own gloo world over a file store
    world = args.gpus
    wl = WORKLOADS[args.workload]
    res = _run_reference(world, args.steps, max(3, args.warmup), args.workload, max(2.0, args.min_seconds))
    desc = _describe_reference(res, args.workload)
    value = desc['value']
    steps = res['steps']
    line = {
        'impl': 'reference', 'metric': wl['metric'], 'value': value, 'unit': 'samples/s', 'n_gpus': world,
        'steps': steps, 'warmup': max(3, args.warmup),
        'ms_per_step': round(steps * wl['batch'] * world / max(value, 1e-9) / steps * 1e3, 4),
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': wl['name'].split(',')[0] + ' — reference CPU path: DDP over gloo on the host cores, fp32, '
                               f'{wl["batch"]} samples/rank/step, metrics reduced once per epoch (stock behaviour)',
                   'global_batch': wl['batch'] * world, 'parallelism': f'dp{world}',
                   'threads_per_rank': res['threads_per_rank'], 'thread_calibration': res.get('calibration'),
                   'timing': f'median of {res.get("windows", 1)} windows of {steps} steps, wall clock of train_epoch, max over ranks'},
        'cpu_baseline': desc,
        'per_step_reduce_value': desc['per_step_reduce_value'],
        'e2e': {'value': value, 'unit': 'samples/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }
    print(json.dumps(line), file=JSON_OUT, flush=True)


def _claim_stdout():
    """The contract is ONE JSON line on stdout.  Libraries (NCCL's version banner, cuDNN warnings) write to fd 1 too, so
    fd 1 is pointed at stderr for the whole run and the JSON line goes to the saved original descriptor."""
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    return os.fdopen(saved, 'w')


if __name__ == '__main__':
    a = parse_args()
    JSON_OUT = _claim_stdout()
    if a.impl == 'reference':
        reference_arm(a)
    else:
        native_arm(a)
