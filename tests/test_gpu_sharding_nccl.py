"""N > 1 on real GPUs (SURVEY §8e, config 5's optional gather): every rank runs its contiguous channel shard through the C ABI on
its own GPU — no data-path collective — and shard.gather_audio / gather_spectra reassemble the shards over NCCL. The gathered result
must equal, byte for byte, what ONE GPU computes for all channels. Skipped when fewer than two GPUs are visible."""
import os
import sys

import numpy as np
import pytest

torch = pytest.importorskip("torch")
import torch.distributed as dist  # noqa: E402
import torch.multiprocessing as mp  # noqa: E402

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


def _worker(rank, world, port, C, T, chain, ret):
    sys.path.insert(0, HERE); sys.path.insert(0, os.path.dirname(HERE))
    import selenite_lite_b200 as slb
    os.environ["MASTER_ADDR"] = "127.0.0.1"; os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    lo, hi = slb.shard.shard_range(C, rank, world)
    x = torch.from_numpy(slb.synth_iq(hi - lo, T, first_channel=lo)).cuda(rank)   # each rank synthesises only its own channels
    d = slb.DspIf(hi - lo, chain=chain, device=rank)
    y = d.rx_process(x)
    full = slb.shard.gather_audio(y, C)                                            # NCCL all-gather (int32 frames)
    spec = slb.shard.gather_spectra(d.spectrum(x[:, :512].contiguous()), C) if chain == slb.CHAIN_RX_SSB_F32 else None
    torch.cuda.synchronize()
    assert dist.get_backend() == "nccl" and full.is_cuda and full.shape == (C, T, 2)
    if rank == 0:
        ret["full"] = full.cpu().numpy().copy()
        if spec is not None:
            ret["spec"] = spec.cpu().numpy().copy()
    dist.barrier(); dist.destroy_process_group()


@pytest.mark.parametrize("chain_name", ["rx_f32", "rx_q15"])
@pytest.mark.parametrize("C", [21, 32])      # 21: shards of 10 and 11 (padded gather); 32: equal shards (one all-gather into the result)
def test_two_gpu_shards_gather_over_nccl(C, chain_name):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    sys.path.insert(0, HERE)
    import selenite_lite_b200 as slb
    chain = slb.CHAIN_RX_SSB_F32 if chain_name == "rx_f32" else slb.CHAIN_RX_SSB_Q15
    T = 1536 * 2
    mgr = mp.Manager(); ret = mgr.dict()
    mp.spawn(_worker, args=(2, 29500 + os.getpid() % 2000, C, T, chain, ret), nprocs=2, join=True)
    xw = torch.from_numpy(slb.synth_iq(C, T)).cuda(0)
    d = slb.DspIf(C, chain=chain, device=0)
    whole = d.rx_process(xw).cpu().numpy()
    assert np.array_equal(ret["full"], whole)
    if chain == slb.CHAIN_RX_SSB_F32:
        assert np.array_equal(ret["spec"], d.spectrum(xw[:, :512].contiguous()).cpu().numpy())
