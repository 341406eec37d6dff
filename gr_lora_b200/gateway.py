"""The gateway receiver over the C ABI (lora_b200_gateway_*, SURVEY.md 8f N4): wideband IQ in, chunk by chunk, the frames of
every (channel, spreading factor) out, one call per chunk.

The channelizer (``channelizer``) filters every channel of ``channel_list`` and one decoder per SF (``decoder`` with
``n_streams = len(channel_list)``) runs on all channels; between them the IQ stays in device memory, and what a stream did
not consume in one call is presented again in the next.  Each (channel, SF) stream decodes exactly what the channelizer
followed by a single-stream decoder on that channel decodes."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _native as N
from .decoder import _dev_ptr, decoder

FRAME_DTYPE = np.dtype([("channel", "<u4"), ("sf", "<u4")] +
                       [(n, decoder.FRAME_DTYPE.fields[n][0]) for n in decoder.FRAME_DTYPE.names])


def _sf_mask(sfs) -> int:
    return sum(1 << int(s) for s in set(sfs))


class gateway:
    """gateway(samp_rate, center_freq, channel_list, bandwidth, sfs, ...): ``decimation`` divides the wideband rate down to
    the decoders' rate (lora_receiver's rule); ``reduced_rate`` is the SFs that use reduced rate (None: LoRa's default at
    125 kHz, SF11 and SF12); ``conj`` conjugates the channel samples (lora_receiver(conj=True)); ``max_in_per_call`` wideband
    items per work() call at most (0 = 1 << 22); ``max_frames_per_call`` per (channel, SF) stream (0 = 8)."""

    FRAME_DTYPE = FRAME_DTYPE

    def __init__(self, samp_rate, center_freq, channel_list, bandwidth, sfs=(7, 8, 9, 10, 11, 12), implicit=False, cr=4, crc=True,
                 decimation=1, reduced_rate=None, conj=False, demod="gradient", device=-1, max_in_per_call=0, max_frames_per_call=0,
                 disable_drift_correction=False):
        self._L = N.lib()
        self._h = None
        self.channel_list = [float(f) for f in channel_list]
        self._cl = (C.c_float * max(len(self.channel_list), 1))(*self.channel_list)
        demod_id = {"gradient": N.DEMOD_GRADIENT, "fft": N.DEMOD_FFT}[demod] if isinstance(demod, str) else int(demod)
        self.sfs = sorted(set(int(s) for s in sfs))
        cfg = N.GatewayConfig(samp_rate=float(samp_rate), center_freq=float(center_freq),
                              channel_list=C.cast(self._cl, C.POINTER(C.c_float)) if self.channel_list else None,
                              n_channels=len(self.channel_list), bandwidth=int(bandwidth), decimation=int(decimation),
                              sf_mask=_sf_mask(sfs), reduced_rate_mask=0 if reduced_rate is None else _sf_mask(reduced_rate),
                              implicit=int(bool(implicit)), cr=int(cr), crc=int(bool(crc)), demod=demod_id, conj=int(bool(conj)),
                              disable_drift_correction=int(bool(disable_drift_correction)), device=int(device),
                              max_in_per_call=int(max_in_per_call), max_frames_per_call=int(max_frames_per_call))
        self.cfg = cfg
        h = self._L.lora_b200_gateway_create(C.byref(cfg))
        if not h:
            raise RuntimeError("lora_b200_gateway_create failed: " + self._L.lora_b200_last_error().decode(errors="replace"))
        self._h = h
        self.decimation = int(decimation)
        self.max_in_per_call = int(max_in_per_call) or (1 << 22)

    def close(self):
        if self._h:
            self._L.lora_b200_gateway_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def work(self, x) -> np.ndarray:
        """One chunk of wideband IQ: a host complex64 array or a device tensor (its length a multiple of the decimation).
        Returns the frames decoded in the call (FRAME_DTYPE), ordered by (sf, channel, seq)."""
        if getattr(x, "is_cuda", True) is False:          # a host torch tensor
            x = x.numpy()
        if isinstance(x, np.ndarray):
            a = np.ascontiguousarray(x, dtype=np.complex64).reshape(-1)
            ptr, n, host = a.ctypes.data, a.size, 1
        else:
            ptr, n, host = _dev_ptr(x), int(x.numel()), 0
        nf = C.c_size_t(0)
        N.check(self._L.lora_b200_gateway_work(self._h, ptr, n, host, C.byref(nf)), "lora_b200_gateway_work")
        fp = C.c_void_p(0)
        n = int(self._L.lora_b200_gateway_frames_last(self._h, C.byref(fp)))
        if n == 0:
            return np.zeros(0, FRAME_DTYPE)
        return np.frombuffer(C.string_at(fp.value, n * FRAME_DTYPE.itemsize), dtype=FRAME_DTYPE).copy()

    def run(self, capture, chunk_items=None) -> np.ndarray:
        """A whole host capture, chunk by chunk (chunk_items wideband items, default max_in_per_call, rounded down to a
        multiple of the decimation); a tail shorter than the decimation is dropped.  Returns all frames in call order."""
        x = np.ascontiguousarray(capture, dtype=np.complex64).reshape(-1)
        step = min(int(chunk_items or self.max_in_per_call), self.max_in_per_call)
        step -= step % self.decimation
        if step <= 0:
            raise ValueError("chunk_items must be at least the decimation")
        end = x.size - x.size % self.decimation
        out = [self.work(x[p:min(p + step, end)]) for p in range(0, end, step)]
        return np.concatenate(out) if out else np.zeros(0, FRAME_DTYPE)

    def reset(self):
        """Decoders and channelizer back to the state of a fresh gateway."""
        N.check(self._L.lora_b200_gateway_reset(self._h), "lora_b200_gateway_reset")

    def position(self, channel, sf):
        """(items of the channel consumed by the SF's decoder since creation / reset, items held over for the next call)"""
        consumed, pending = C.c_uint64(0), C.c_uint32(0)
        N.check(self._L.lora_b200_gateway_position(self._h, int(channel), int(sf), C.byref(consumed), C.byref(pending)),
                "lora_b200_gateway_position")
        return int(consumed.value), int(pending.value)

    def timing(self) -> dict:
        """Device time of the last work() call in ms, from CUDA events."""
        ms = (C.c_float * 4)()
        N.check(self._L.lora_b200_gateway_timing(self._h, ms, 4), "lora_b200_gateway_timing")
        return dict(zip(("h2d", "channelizer", "gather", "decoders"), (float(v) for v in ms)))
