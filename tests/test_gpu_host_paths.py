"""The channel-group pipeline of the host bulk path (PASS chain, channelizer): batches wide enough for more groups than there are
staging slots, so the slot streams wrap and a slot's buffers are reused while the pipeline runs."""
import numpy as np
import pytest

import selenite_lite_b200 as slb

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu


@pytest.mark.timeout(240, method="thread")
def test_pass_host_path_over_four_channel_groups_is_bit_exact_copy():
    C, T = 10, 1 << 22                                      # 16 MiB per channel: groups of 3 channels under the 48 MiB cap -> 4 groups
    x = np.random.default_rng(5).integers(-32768, 32767, (C, T, 2), dtype=np.int16, endpoint=True)
    d = slb.DspIf(C, chain=slb.CHAIN_PASS)
    for rep in range(2):
        assert np.array_equal(d.rx_process(x), x)
    assert d.kernel_launches() == 2 * 4                     # one copy kernel per group


@pytest.mark.timeout(240, method="thread")
def test_chan64_host_path_over_four_stream_groups_matches_device_path():
    S, T = 200, 768 * 256                                   # 768 KiB per stream: groups of 64 streams -> 4 groups
    rng = np.random.default_rng(6)
    x = [rng.integers(-12000, 12000, (S, T, 2), dtype=np.int16) for _ in range(2)]
    host = slb.DspIf(S, fs=192000, chain=slb.CHAIN_CHAN64_F32)
    dev = slb.DspIf(S, fs=192000, chain=slb.CHAIN_CHAN64_F32)
    for xi in x:                                            # two calls: the carried state crosses the group cuts as well
        y = dev.chan_process(torch.from_numpy(xi).cuda()); torch.cuda.synchronize()
        assert np.array_equal(host.chan_process(xi), y.cpu().numpy())
