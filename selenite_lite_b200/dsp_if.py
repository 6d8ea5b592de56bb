"""Host-side mirror of the reference module Core/Src/dsp_if.c, batched over channels.

Method names, argument order and the unit of `size` are the firmware's (Core/Inc/dsp_if.h:42-51); every method is
one call into the C ABI (include/selenite_b200.h). numpy arrays are host buffers ([channels][size] as in the C ABI),
torch CUDA tensors go through the device bulk path.
"""
import ctypes as C

import numpy as np

from . import _lib

CHAIN_PASS, CHAIN_RX_SSB_F32, CHAIN_TX_SSB_F32, CHAIN_CHAN64_F32, CHAIN_RX_SSB_Q15, CHAIN_TX_F32 = 0, 1, 2, 3, 4, 5
MODE_LSB, MODE_USB, MODE_CW, MODE_CWR, MODE_AM, MODE_FM, MODE_DIG, MODE_PKT = 0x00, 0x01, 0x02, 0x03, 0x04, 0x08, 0x0A, 0x0C
RX_PATH_AUTO, RX_PATH_FFT = 0, 1


class SeleniteError(RuntimeError):
    pass


def default_rx_f32_params(fs=48000):
    p = _lib.RxF32Params()
    rc = _lib.load().slb_default_rx_f32_params(fs, C.byref(p))
    if rc:
        raise SeleniteError("slb_default_rx_f32_params -> %d" % rc)
    return p


def default_tx_f32_params(fs=48000):
    p = _lib.TxF32Params()
    rc = _lib.load().slb_default_tx_f32_params(fs, C.byref(p))
    if rc:
        raise SeleniteError("slb_default_tx_f32_params -> %d" % rc)
    return p


def tx_params_to_dict(p, mask):
    return dict(fft_len=p.fft_len, hop=p.hop, alc_block=p.alc_block, alc_target=p.alc_target, alc_decay=p.alc_decay,
                alc_floor=p.alc_floor, alc_gmax=p.alc_gmax, mask=mask)


def default_tx_mod_params(fs=48000):
    p = _lib.TxModParams()
    rc = _lib.load().slb_default_tx_mod_params(fs, C.byref(p))
    if rc:
        raise SeleniteError("slb_default_tx_mod_params -> %d" % rc)
    return p


def tx_mod_params_to_dict(tx, mod, mask, fs, mode):
    """The AM / FM transmit chain as plain data (the oracle's tx_mod_f32 parameters): `tx` the ALC, `mod` the modulator constants."""
    return dict(fft_len=tx.fft_len, hop=tx.hop, alc_block=tx.alc_block, fs=fs, alc_decay=tx.alc_decay, alc_floor=tx.alc_floor,
                alc_gmax=tx.alc_gmax, mask=mask, modulator=1 if mode == MODE_AM else 2, am_carrier=mod.am_carrier,
                am_depth=mod.am_depth, fm_deviation_hz=mod.fm_deviation_hz, fm_level=mod.fm_level)


def default_chan_params(fs=192000):
    p = _lib.ChanParams()
    rc = _lib.load().slb_default_chan_params(fs, C.byref(p))
    if rc:
        raise SeleniteError("slb_default_chan_params -> %d" % rc)
    return p


def chan_params_to_dict(p):
    return dict(bins=p.bins, taps_per_branch=p.taps_per_branch, agc_block=p.agc_block, envelope=p.envelope,
                agc_target=p.agc_target, agc_decay=p.agc_decay, agc_floor=p.agc_floor, agc_gmax=p.agc_gmax,
                proto=np.array(p.proto[:p.bins * p.taps_per_branch], np.float32))


def default_rx_q15_params(fs=48000):
    p = _lib.RxQ15Params()
    rc = _lib.load().slb_default_rx_q15_params(fs, C.byref(p))
    if rc:
        raise SeleniteError("slb_default_rx_q15_params -> %d" % rc)
    return p


def q15_params_to_dict(p, lsb=0):
    return dict(ntaps=p.ntaps, agc_block=p.agc_block, agc_window=p.agc_window, lsb=int(lsb),
                taps_i=np.array(p.taps_i[:], np.int16), taps_q=np.array(p.taps_q[:], np.int16), rel=np.array(p.rel[:], np.int16),
                agc_target=p.agc_target, agc_floor=p.agc_floor, agc_gmax_q15=p.agc_gmax_q15,
                bq_stages=p.bq_stages, bq_postshift=p.bq_postshift, bq_coeffs=np.array(p.bq_coeffs[:], np.int16))


def default_mask(fs=48000, fft_len=512, mode=MODE_USB):
    m = np.zeros(2 * fft_len, np.float32)
    rc = _lib.load().slb_default_mask(fs, fft_len, mode, m.ctypes.data)
    if rc:
        raise SeleniteError("slb_default_mask -> %d" % rc)
    return m.view(np.complex64)


def params_to_dict(p, mask):
    """The chain parameters as plain data (what a test hands to the oracle)."""
    return dict(fft_len=p.fft_len, hop=p.hop, agc_block=p.agc_block,
                biquad=np.array(p.biquad[:5 * p.n_stages], np.float32).reshape(-1, 5),
                agc_target=p.agc_target, agc_decay=p.agc_decay, agc_floor=p.agc_floor, agc_gmax=p.agc_gmax, mask=mask)


class LiveFeeder:
    """slb_live_*: chunks of `ticks_per_chunk` ms through a three-stream pipeline (copy in | chain + ring replay | copy out)."""

    def __init__(self, dsp, ticks_per_chunk, depth, rx, tx):
        self.dsp, self.rx, self.tx = dsp, bool(rx), bool(tx)
        self.frames = ticks_per_chunk * dsp.block_frames
        self.h = C.c_void_p()
        dsp._ck(dsp.lib.slb_live_open(dsp.h, ticks_per_chunk, depth, int(rx), int(tx), C.byref(self.h)), "live_open")

    def push(self, adc=None, usb_out=None):
        keep = []
        def ptr(a):
            if a is None:
                return None
            a = np.ascontiguousarray(a, np.int16); assert a.shape == (self.dsp.channels, self.frames, 2); keep.append(a); return a.ctypes.data
        self.dsp._ck(self.dsp.lib.slb_live_push(self.h, ptr(adc), ptr(usb_out)), "live_push")

    def pop(self):
        """Returns (usb_in, dac, latency_us) of the oldest chunk in flight."""
        shape = (self.dsp.channels, self.frames, 2)
        usb_in = np.zeros(shape, np.int16) if self.rx else None; dac = np.zeros(shape, np.int16) if self.tx else None
        lat = C.c_float()
        self.dsp._ck(self.dsp.lib.slb_live_pop(self.h, usb_in.ctypes.data if self.rx else None, dac.ctypes.data if self.tx else None, C.byref(lat)), "live_pop")
        return usb_in, dac, lat.value

    def in_flight(self):
        return self.dsp.lib.slb_live_in_flight(self.h)

    def close(self):
        if self.h:
            self.dsp.lib.slb_live_close(self.h); self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class DspIf:
    """One context = one GPU's shard of channels."""

    def __init__(self, channels, fs=48000, chain=CHAIN_PASS, device=0):
        self.lib = _lib.load()
        self.channels, self.fs, self.chain, self.device = int(channels), int(fs), int(chain), int(device)
        cfg = _lib.Config(self.channels, self.fs, self.device, self.chain)
        h = C.c_void_p()
        rc = self.lib.slb_create(C.byref(cfg), C.byref(h))
        if rc:
            raise SeleniteError("slb_create -> %d: %s" % (rc, self.lib.slb_last_error(None).decode()))
        self.h = h
        self.block_frames = self.fs // 1000
        self.ring_frames = 8 * self.block_frames

    def close(self):
        if getattr(self, "h", None):
            self.lib.slb_destroy(self.h)
            self.h = None

    __del__ = close

    def _ck(self, rc, what):
        if rc:
            raise SeleniteError("%s -> %d: %s" % (what, rc, self.lib.slb_last_error(self.h).decode()))

    # ---- firmware API (dsp_if.h:42-51) ----
    def DSP_Init(self): self._ck(self.lib.SLB_DSP_Init(self.h), "DSP_Init")
    def DSP_Set_RX(self): self._ck(self.lib.SLB_DSP_Set_RX(self.h), "DSP_Set_RX")
    def DSP_Set_TX(self): self._ck(self.lib.SLB_DSP_Set_TX(self.h), "DSP_Set_TX")

    def DSP_Set_Mode(self, mode, channel=None):
        if channel is None:
            self._ck(self.lib.SLB_DSP_Set_Mode(self.h, mode), "DSP_Set_Mode")
        else:
            self._ck(self.lib.SLB_DSP_Set_Mode_Channel(self.h, channel, mode), "DSP_Set_Mode_Channel")

    def DSP_In_Buff_Write(self, pbuf, size=None):
        """pbuf int16/uint16 [channels][size]; size = half-words per channel (2 per frame)."""
        a = np.ascontiguousarray(pbuf).view(np.int16).reshape(self.channels, -1)
        size = a.shape[1] if size is None else size
        self._ck(self.lib.SLB_DSP_In_Buff_Write(self.h, a.ctypes.data, size), "DSP_In_Buff_Write")

    def DSP_In_Buff_Read(self, size):
        """size = bytes per channel (4 per frame). Returns int16 [channels][size/2]."""
        out = np.zeros((self.channels, size // 2), np.int16)
        self._ck(self.lib.SLB_DSP_In_Buff_Read(self.h, out.ctypes.data, size), "DSP_In_Buff_Read")
        return out

    def DSP_Out_Buff_Write(self, pbuf, size=None):
        """pbuf int16 [channels][n]; size = BYTES per channel."""
        a = np.ascontiguousarray(pbuf).view(np.int16).reshape(self.channels, -1)
        size = a.shape[1] * 2 if size is None else size
        self._ck(self.lib.SLB_DSP_Out_Buff_Write(self.h, a.ctypes.data, size), "DSP_Out_Buff_Write")

    def DSP_Out_Buff_Read(self, size):
        """size = half-words per channel. Returns int16 [channels][size]."""
        out = np.zeros((self.channels, size), np.int16)
        self._ck(self.lib.SLB_DSP_Out_Buff_Read(self.h, out.ctypes.data, size), "DSP_Out_Buff_Read")
        return out

    def DSP_Out_Buff_Mute(self): self._ck(self.lib.SLB_DSP_Out_Buff_Mute(self.h), "DSP_Out_Buff_Mute")

    # ---- per-channel cadence (SLB_DSP_*_Ch): `active` uint8[channels], 0 = this channel's producer / consumer did not fire
    @staticmethod
    def _mask(active):
        if active is None:
            return None, None
        a = np.ascontiguousarray(active, np.uint8)
        return a, a.ctypes.data

    def DSP_In_Buff_Write_Ch(self, pbuf, active=None):
        a = np.ascontiguousarray(pbuf).view(np.int16).reshape(self.channels, -1); keep, m = self._mask(active)
        self._ck(self.lib.SLB_DSP_In_Buff_Write_Ch(self.h, a.ctypes.data, a.shape[1], m), "DSP_In_Buff_Write_Ch")

    def DSP_In_Buff_Read_Ch(self, size, active=None):
        out = np.zeros((self.channels, size // 2), np.int16); keep, m = self._mask(active)
        self._ck(self.lib.SLB_DSP_In_Buff_Read_Ch(self.h, out.ctypes.data, size, m), "DSP_In_Buff_Read_Ch")
        return out

    def DSP_Out_Buff_Write_Ch(self, pbuf, active=None):
        a = np.ascontiguousarray(pbuf).view(np.int16).reshape(self.channels, -1); keep, m = self._mask(active)
        self._ck(self.lib.SLB_DSP_Out_Buff_Write_Ch(self.h, a.ctypes.data, a.shape[1] * 2, m), "DSP_Out_Buff_Write_Ch")

    def DSP_Out_Buff_Read_Ch(self, size, active=None):
        out = np.zeros((self.channels, size), np.int16); keep, m = self._mask(active)
        self._ck(self.lib.SLB_DSP_Out_Buff_Read_Ch(self.h, out.ctypes.data, size, m), "DSP_Out_Buff_Read_Ch")
        return out

    def DSP_Set_Sidetone(self, freq_hz, level):
        self._ck(self.lib.SLB_DSP_Set_Sidetone(self.h, int(freq_hz), float(level)), "DSP_Set_Sidetone")

    def DSP_Key(self, key_down=None):
        """key_down: per-channel booleans (None = all keys up)."""
        if key_down is None:
            self._ck(self.lib.SLB_DSP_Key(self.h, None), "DSP_Key"); return
        k = np.ascontiguousarray(np.asarray(key_down).astype(np.uint8)); assert k.size == self.channels
        self._ck(self.lib.SLB_DSP_Key(self.h, k.ctypes.data), "DSP_Key")

    def direction(self):
        return self.lib.slb_get_direction(self.h)

    def feeder_run(self, adc=None, usb_out=None):
        """Replay `ticks` firmware milliseconds in one call (slb_feeder_run): adc / usb_out int16 [channels][ticks*block][2]
        host streams (either may be None). Returns (usb_in, dac) of the same shape (None for a skipped direction)."""
        io = _lib.FeederIo(); keep = []
        ticks = None
        usb_in = dac = None
        if adc is not None:
            adc = np.ascontiguousarray(adc, np.int16); usb_in = np.zeros_like(adc); keep += [adc, usb_in]
            io.adc, io.usb_in = adc.ctypes.data, usb_in.ctypes.data; ticks = adc.shape[1] // self.block_frames
        if usb_out is not None:
            usb_out = np.ascontiguousarray(usb_out, np.int16); dac = np.zeros_like(usb_out); keep += [usb_out, dac]
            io.usb_out, io.dac = usb_out.ctypes.data, dac.ctypes.data
            if ticks is not None and usb_out.shape[1] // self.block_frames != ticks:
                raise ValueError("feeder_run: adc and usb_out must cover the same number of ticks")
            ticks = usb_out.shape[1] // self.block_frames
        for a in (adc, usb_out):
            if a is not None and (a.shape[0] != self.channels or a.shape[1] % self.block_frames != 0 or a.shape[2] != 2):
                raise ValueError("feeder_run: streams are int16 [channels][ticks * block_frames][2]")
        if ticks is None:
            raise ValueError("feeder_run: no stream given")
        self._ck(self.lib.slb_feeder_run(self.h, C.byref(io), ticks), "feeder_run")
        return usb_in, dac

    def live_open(self, ticks_per_chunk, depth=3, rx=True, tx=True):
        """Live feeder (slb_live_*): returns a LiveFeeder bound to this context."""
        return LiveFeeder(self, ticks_per_chunk, depth, rx, tx)

    def AUDIO_AudioCmd(self, pbuf, size, cmd):
        a = np.ascontiguousarray(pbuf)
        self._ck(self.lib.SLB_AUDIO_AudioCmd(self.h, a.ctypes.data, size, cmd), "AUDIO_AudioCmd")
        return a

    def ring_ptrs_channel(self, channel, which=0):
        o = (C.c_uint32 * 3)()
        self._ck(self.lib.slb_ring_get_ptrs_channel(self.h, which, channel, C.byref(o)), "ring_get_ptrs_channel")
        return tuple(o)

    def ring_ptrs(self, which=0):
        o = (C.c_uint32 * 3)()
        self._ck(self.lib.slb_ring_get_ptrs(self.h, which, C.byref(o)), "ring_get_ptrs")
        return tuple(o)

    def ring_iq(self, which=0):
        i = np.zeros((self.channels, self.ring_frames), np.int16); q = np.zeros_like(i)
        self._ck(self.lib.slb_ring_get_iq(self.h, which, i.ctypes.data, q.ctypes.data), "ring_get_iq")
        return i, q

    # ---- chain parameters ----
    def rx_params(self):
        p = _lib.RxF32Params()
        self._ck(self.lib.slb_get_rx_f32_params(self.h, C.byref(p)), "get_rx_f32_params")
        return p

    def set_rx_params(self, p): self._ck(self.lib.slb_set_rx_f32_params(self.h, C.byref(p)), "set_rx_f32_params")

    def set_rx_path(self, path):
        """RX_PATH_AUTO (tensor-core FIR kernel where the mask allows) or RX_PATH_FFT (FFT kernel for every channel)."""
        self._ck(self.lib.slb_set_rx_path(self.h, int(path)), "set_rx_path")

    def mask(self, mode=MODE_USB):
        m = np.zeros(2 * self.rx_params().fft_len, np.float32)
        self._ck(self.lib.slb_get_mask(self.h, mode, m.ctypes.data), "get_mask")
        return m.view(np.complex64)

    def set_mask(self, mode, mask):
        m = np.ascontiguousarray(np.asarray(mask, np.complex64)).view(np.float32)
        self._ck(self.lib.slb_set_mask(self.h, mode, m.ctypes.data), "set_mask")

    def tx_params(self):
        p = _lib.TxF32Params()
        self._ck(self.lib.slb_get_tx_f32_params(self.h, C.byref(p)), "get_tx_f32_params")
        return p

    def set_tx_params(self, p): self._ck(self.lib.slb_set_tx_f32_params(self.h, C.byref(p)), "set_tx_f32_params")

    def tx_mod_params(self):
        """AM / FM modulator constants of a CHAIN_TX_F32 context."""
        p = _lib.TxModParams()
        self._ck(self.lib.slb_get_tx_mod_params(self.h, C.byref(p)), "get_tx_mod_params")
        return p

    def set_tx_mod_params(self, p): self._ck(self.lib.slb_set_tx_mod_params(self.h, C.byref(p)), "set_tx_mod_params")

    def set_phase_tap(self, phase=None):
        """CHAIN_TX_F32: phase = torch CUDA int32/uint32 [channels][frames] receiving the FM phase accumulator (2^-32 turn) after each
        sample of FM channels on the next tx_process calls (None switches the tap off)."""
        self._keep_phase = phase
        self._ck(self.lib.slb_tx_set_phase_tap(self.h, phase.data_ptr() if phase is not None else None), "tx_set_phase_tap")

    def chan_params(self):
        p = _lib.ChanParams()
        self._ck(self.lib.slb_get_chan_params(self.h, C.byref(p)), "get_chan_params")
        return p

    def set_chan_params(self, p): self._ck(self.lib.slb_set_chan_params(self.h, C.byref(p)), "set_chan_params")

    def rx_q15_params(self):
        p = _lib.RxQ15Params()
        self._ck(self.lib.slb_get_rx_q15_params(self.h, C.byref(p)), "get_rx_q15_params")
        return p

    def set_rx_q15_params(self, p): self._ck(self.lib.slb_set_rx_q15_params(self.h, C.byref(p)), "set_rx_q15_params")

    def set_q15_debug_taps(self, audio=None, gain=None):
        """audio: torch CUDA int16 [channels][frames]; gain: torch CUDA int32 [channels][frames/48] (Q15 gain per block)."""
        self._keep_taps = (audio, gain)
        self._ck(self.lib.slb_rx_q15_set_debug_taps(self.h, audio.data_ptr() if audio is not None else None,
                                                    gain.data_ptr() if gain is not None else None), "rx_q15_set_debug_taps")

    def oracle_params(self, mode=MODE_USB):
        if self.chain == CHAIN_RX_SSB_Q15:
            return q15_params_to_dict(self.rx_q15_params(), lsb=mode in (MODE_LSB, MODE_CWR))
        if self.chain == CHAIN_CHAN64_F32:
            return chan_params_to_dict(self.chan_params())
        if self.chain == CHAIN_TX_F32 and mode in (MODE_AM, MODE_FM):
            return tx_mod_params_to_dict(self.tx_params(), self.tx_mod_params(), self.mask(mode), self.fs, mode)
        if self.chain in (CHAIN_TX_SSB_F32, CHAIN_TX_F32):
            return tx_params_to_dict(self.tx_params(), self.mask(mode))
        prm = params_to_dict(self.rx_params(), self.mask(mode))
        prm["envelope"] = 1 if mode == MODE_AM else 2 if mode == MODE_FM else 0   # the oracle chain's detector: Re, |z| (AM), limiter-discriminator (FM)
        return prm

    # ---- bulk path ----
    def rx_process(self, x, out=None, stream=None, _dir="rx"):
        """x: torch CUDA int16 tensor [channels][frames][2] (device path, async on `stream`/current stream) or
        numpy int16 array of that shape (host path, synchronous). Returns `out`."""
        if isinstance(x, np.ndarray):
            x = np.ascontiguousarray(x, np.int16)
            frames = x.shape[1]
            out = np.empty_like(x) if out is None else out
            self._ck(getattr(self.lib, "slb_%s_process_host" % _dir)(self.h, x.ctypes.data, out.ctypes.data, frames), _dir + "_process_host")
            return out
        import torch
        assert x.is_cuda and x.dtype == torch.int16 and x.is_contiguous() and x.shape[0] == self.channels
        frames = x.shape[1]
        out = torch.empty_like(x) if out is None else out
        s = torch.cuda.current_stream(x.device).cuda_stream if stream is None else stream
        self._ck(getattr(self.lib, "slb_%s_process_device" % _dir)(self.h, x.data_ptr(), out.data_ptr(), frames, s), _dir + "_process_device")
        return out

    def tx_process(self, x, out=None, stream=None):
        """TX direction (context created with CHAIN_TX_SSB_F32 or CHAIN_TX_F32): mic frames (L = R) in, modulated I/Q frames out."""
        return self.rx_process(x, out, stream, _dir="tx")

    def chan_process(self, x, out=None, stream=None):
        """Channelizer (context created with CHAIN_CHAN64_F32): x int16 [streams][frames][2] wideband I/Q ->
        int16 [streams][64][frames/64][2] demodulated narrowband audio (L = R), channel-major."""
        if isinstance(x, np.ndarray):
            x = np.ascontiguousarray(x, np.int16)
            frames = x.shape[1]
            out = np.empty((x.shape[0], 64, frames // 64, 2), np.int16) if out is None else out
            self._ck(self.lib.slb_chan_process_host(self.h, x.ctypes.data, out.ctypes.data, frames), "chan_process_host")
            return out
        import torch
        assert x.is_cuda and x.dtype == torch.int16 and x.is_contiguous() and x.shape[0] == self.channels
        frames = x.shape[1]
        out = torch.empty((x.shape[0], 64, frames // 64, 2), dtype=torch.int16, device=x.device) if out is None else out
        s = torch.cuda.current_stream(x.device).cuda_stream if stream is None else stream
        self._ck(self.lib.slb_chan_process_device(self.h, x.data_ptr(), out.data_ptr(), frames, s), "chan_process_device")
        return out

    def chan_process_pinned(self, x_pinned, out_pinned):
        self._ck(self.lib.slb_chan_process_host(self.h, x_pinned.data_ptr(), out_pinned.data_ptr(), x_pinned.shape[1]), "chan_process_host")
        return out_pinned

    def rx_process_pinned(self, x_pinned, out_pinned):
        """torch pinned host tensors [channels][frames][2]; chunked H2D / kernel / D2H overlap inside the library."""
        frames = x_pinned.shape[1]
        self._ck(self.lib.slb_rx_process_host(self.h, x_pinned.data_ptr(), out_pinned.data_ptr(), frames), "rx_process_host")
        return out_pinned

    def spectrum(self, x, out=None, stream=None):
        """Power spectrum of x = int16 [channels][N][2] (CUDA tensor): float32 [channels][N], natural bin order."""
        import torch
        assert x.is_cuda and x.is_contiguous() and x.dtype == torch.int16
        n = x.shape[1]
        if out is None:
            out = torch.empty((x.shape[0], n), dtype=torch.float32, device=x.device)
        st = torch.cuda.current_stream().cuda_stream if stream is None else stream
        self._ck(self.lib.slb_rx_spectrum_device(self.h, x.data_ptr(), out.data_ptr(), n, st), "rx_spectrum_device")
        return out

    def set_debug_taps(self, audio=None, gain=None):
        self._keep_taps = (audio, gain)
        self._ck(self.lib.slb_rx_set_debug_taps(self.h, audio.data_ptr() if audio is not None else None,
                                                gain.data_ptr() if gain is not None else None), "set_debug_taps")

    # ---- stage library (slb_st_*): torch CUDA tensors = device arrays [channels][n], numpy arrays = host coefficients ----
    def st(self, name, *args, stream=None):
        conv, keep = [], []
        for a in args:
            if isinstance(a, np.ndarray):
                a = np.ascontiguousarray(a); keep.append(a); conv.append(a.ctypes.data)
            elif hasattr(a, "data_ptr"):
                assert a.is_cuda and a.is_contiguous(); conv.append(a.data_ptr())
            else:
                conv.append(a)
        self._ck(getattr(self.lib, "slb_st_" + name)(self.h, *conv, stream), "slb_st_" + name)

    # ---- checkpoint ----
    def state_save(self):
        n = C.c_size_t()
        self._ck(self.lib.slb_state_size(self.h, C.byref(n)), "state_size")
        buf = np.zeros(n.value, np.uint8)
        self._ck(self.lib.slb_state_save(self.h, buf.ctypes.data, n.value), "state_save")
        return buf

    def state_load(self, buf):
        buf = np.ascontiguousarray(buf, np.uint8)
        self._ck(self.lib.slb_state_load(self.h, buf.ctypes.data, buf.size), "state_load")

    def kernel_launches(self): return int(self.lib.slb_kernel_launches(self.h))
    def sync(self): self._ck(self.lib.slb_sync(self.h), "sync")
