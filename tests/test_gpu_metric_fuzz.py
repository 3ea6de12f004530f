"""The differential fuzz of tests/test_metric_fuzz_vs_reference.py with the PRODUCT in the loop: libdmlb's device slab (K3 fold,
K4 reduce / peer exchange) replays the same seeded random sessions the unmodified reference replayed (its answers are stored
in tests/golden/metric_fuzz_w*.json) and must agree with it within SURVEY §8d's tolerances — and with the slab oracle bit
for bit.  World size 2 and 4 run as separate processes sharing the GPU (CUDA-IPC peer mappings, or real NVLink peers on a
multi-GPU box)."""
import json
from pathlib import Path

import pytest
import torch

from helpers import init_gloo, rank_device, spawn
from test_metric_fuzz_vs_reference import run_seeds

pytestmark = pytest.mark.gpu


def test_random_sessions_on_the_device_slab_match_reference_and_oracle_w1():
    from dmlcloud_b200.util.distributed import deinitialize_torch_distributed, init_process_group_dummy

    init_process_group_dummy()
    try:
        assert run_seeds(range(40), 1, 0, device=torch.device('cuda', 0)) > 300
    finally:
        deinitialize_torch_distributed()


def _worker(rank, world, initfile, outdir, first_seed, n_seeds):
    init_gloo(rank, world, initfile)
    import torch.distributed as dist

    from dmlcloud_b200.gradsync import PeerComm

    torch.cuda.set_device(rank_device(rank))
    dev = torch.device('cuda', rank_device(rank))
    comm = PeerComm(dev, None, max_message_bytes=1 << 20)
    checked = run_seeds(range(first_seed, first_seed + n_seeds), world, rank, device=dev, comm=comm)
    Path(outdir, f'ok{rank}.json').write_text(json.dumps({'checked': checked}))
    dist.barrier()
    comm.close()
    dist.destroy_process_group()


@pytest.mark.parametrize('world', [2, 4])
def test_random_sessions_on_the_device_slab_over_the_peer_exchange(world):
    out = spawn(_worker, world, 1000 * world, 10, timeout=600)
    counts = [json.loads((out / f'ok{r}.json').read_text())['checked'] for r in range(world)]
    assert len(set(counts)) == 1 and counts[0] > 80
