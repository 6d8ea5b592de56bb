"""selenite_lite_b200 — B200-native batched implementation of the Selenite Lite sample path
(reference: /root/reference/Core/Src/dsp_if.c). The product is the CUDA shared library behind
include/selenite_b200.h; this package is the thin host-side mirror used by tests, bench and sharded runs."""
from . import _lib
from .dsp_if import (CHAIN_PASS, CHAIN_RX_SSB_F32, CHAIN_TX_SSB_F32, CHAIN_CHAN64_F32, CHAIN_RX_SSB_Q15, CHAIN_TX_F32, RX_PATH_AUTO, RX_PATH_FFT, MODE_AM, MODE_FM, MODE_CW, MODE_CWR, MODE_DIG, MODE_LSB, MODE_PKT, MODE_USB,
                     DspIf, SeleniteError, default_mask, default_rx_f32_params, default_tx_f32_params, default_chan_params, default_rx_q15_params, default_tx_mod_params)
from . import shard, signals
from .signals import channel_tone_hz, synth_fm, synth_iq, synth_mic, synth_wideband

__all__ = ["synth_fm", "DspIf", "SeleniteError", "default_mask", "default_rx_f32_params", "default_tx_f32_params", "synth_iq", "synth_mic", "channel_tone_hz",
           "CHAIN_PASS", "CHAIN_RX_SSB_F32", "CHAIN_TX_SSB_F32", "CHAIN_CHAN64_F32", "CHAIN_RX_SSB_Q15", "CHAIN_TX_F32", "default_tx_mod_params", "RX_PATH_AUTO", "RX_PATH_FFT", "default_rx_q15_params", "MODE_AM", "MODE_FM", "default_chan_params", "synth_wideband", "MODE_LSB", "MODE_USB", "MODE_CW", "MODE_CWR", "MODE_DIG", "MODE_PKT", "_lib"]
