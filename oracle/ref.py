"""ctypes binding of oracle/_ref/liblora_ref.so: the REFERENCE'S OWN lib/decoder_impl.cc, compiled unmodified
against stand-in headers (oracle/ref_wrap.cc, oracle/ref_standins/README.md).  TEST INFRASTRUCTURE ONLY: imported by
tests/, tests/golden/make_golden.py and bench.py's cpu_baseline / --impl reference legs, never by the product.

`RefDecoder` has the interface of `oracle.oracle.Decoder` so the same test bodies run against either; what it cannot
offer is the FFT demodulator inside work(): the reference calls max_frequency_gradient_idx there and leaves
get_shift_fft commented out (lib/decoder_impl.cc:499-500), so `run()` is gradient-mode only while `get_shift_fft`
is available as a stage function.

/root/reference exists only in the build container; `available()` is False where neither it nor a prebuilt
oracle/_ref/liblora_ref.so is present."""
from __future__ import annotations

import ctypes as C
import subprocess
from pathlib import Path

import numpy as np

from .oracle import STEP_DTYPE, Step, _ptr

HERE = Path(__file__).resolve().parent
LIB = HERE / "_ref" / "liblora_ref.so"
REF_ROOT = Path("/root/reference")

_lib = None


def _have_sources() -> bool:
    try:
        return (REF_ROOT / "lib" / "decoder_impl.cc").is_file()
    except OSError:          # a directory the user may not enter: the sources are absent for this user
        return False


def build(force: bool = False) -> Path | None:
    """(Re)build where the reference sources exist; otherwise keep whatever prebuilt file travelled here."""
    if _have_sources():
        if force and LIB.exists():
            LIB.unlink()
        subprocess.run(["make", "-C", str(HERE), "-s", "ref"], check=True)
    return LIB if LIB.exists() else None


def available() -> bool:
    return LIB.exists() or _have_sources()


def lib():
    global _lib
    if _lib is None:
        if build() is None:
            raise RuntimeError("oracle/_ref/liblora_ref.so is not built and /root/reference is absent")
        L = C.CDLL(str(LIB))
        vp, u32, i32, f32, sz = C.c_void_p, C.c_uint32, C.c_int32, C.c_float, C.c_size_t
        L.lr_create.restype = vp
        L.lr_create.argtypes = [f32, u32, C.c_uint8, C.c_int, C.c_uint8, C.c_int, C.c_int, C.c_int]
        L.lr_destroy.argtypes = [vp]
        for n in ("lr_sps", "lr_bins", "lr_bins_hdr", "lr_decim", "lr_delay_after_sync"):
            getattr(L, n).restype = u32
            getattr(L, n).argtypes = [vp]
        L.lr_output_multiple.restype = C.c_int
        L.lr_output_multiple.argtypes = [vp]
        for n in ("lr_bits_per_symbol", "lr_dt"):
            getattr(L, n).restype = C.c_double
            getattr(L, n).argtypes = [vp]
        for n in ("lr_downchirp", "lr_upchirp", "lr_downchirp_ifreq", "lr_upchirp_ifreq", "lr_upchirp_ifreq_v"):
            getattr(L, n).restype = vp
            getattr(L, n).argtypes = [vp]
        L.lr_instantaneous_frequency.argtypes = [vp, vp, vp, u32]
        L.lr_get_shift_fft.restype = u32
        L.lr_get_shift_fft.argtypes = [vp, vp, vp]
        L.lr_get_shift_fft_spectrum.argtypes = [vp, vp, vp]
        L.lr_max_frequency_gradient_idx.restype = u32
        L.lr_max_frequency_gradient_idx.argtypes = [vp, vp]
        L.lr_fine_sync.restype = i32
        L.lr_fine_sync.argtypes = [vp, vp, i32, i32]
        L.lr_detect_preamble_autocorr.restype = f32
        L.lr_detect_preamble_autocorr.argtypes = [vp, vp]
        L.lr_energy_threshold.restype = f32
        L.lr_energy_threshold.argtypes = [vp]
        L.lr_detect_upchirp.restype = f32
        L.lr_detect_upchirp.argtypes = [vp, vp, vp]
        L.lr_detect_downchirp.restype = f32
        L.lr_detect_downchirp.argtypes = [vp, vp]
        L.lr_experimental_determine_cfo.restype = f32
        L.lr_experimental_determine_cfo.argtypes = [vp, vp]
        L.lr_determine_energy.restype = f32
        L.lr_determine_energy.argtypes = [vp, vp]
        L.lr_demod_fft_batch.argtypes = [vp, vp, sz, vp, vp]
        L.lr_demod_grad_batch.argtypes = [vp, vp, sz, vp]
        L.lr_state.restype = C.c_int
        L.lr_state.argtypes = [vp]
        L.lr_work.restype = C.c_int
        L.lr_work.argtypes = [vp, vp, vp]
        L.lr_run.restype = sz
        L.lr_run.argtypes = [vp, vp, sz, vp, sz, vp]
        L.lr_frame_count.restype = sz
        L.lr_frame_count.argtypes = [vp]
        L.lr_frame_len.restype = sz
        L.lr_frame_len.argtypes = [vp, sz]
        L.lr_frame_data.restype = vp
        L.lr_frame_data.argtypes = [vp, sz]
        L.lr_frames_clear.argtypes = [vp]
        L.lr_stdout.restype = C.c_char_p
        L.lr_stdout.argtypes = [vp]
        L.lr_rotl.restype = u32
        L.lr_rotl.argtypes = [u32, u32, u32]
        for n in ("lr_hamming_encode_soft", "lr_hamming_decode_soft_byte"):
            getattr(L, n).restype = C.c_uint8
            getattr(L, n).argtypes = [C.c_uint8]
        L.lr_deinterleave_words.argtypes = [vp, vp, u32, u32, vp]
        L.lr_decode_codewords.restype = sz
        L.lr_decode_codewords.argtypes = [vp, vp, sz, C.c_int, C.c_uint8, vp, sz, vp]
        _lib = L
    return _lib


class RefDecoder:
    """The reference's decoder_impl behind lora::decoder::make's argument list (include/lora/decoder.h:705)."""

    def __init__(self, samp_rate=1e6, bandwidth=125000, sf=7, implicit=False, cr=4, crc=True,
                 reduced_rate=False, disable_drift_correction=False):
        self.L = lib()
        self.h = self.L.lr_create(samp_rate, bandwidth, sf, int(implicit), cr, int(crc), int(reduced_rate),
                                  int(disable_drift_correction))
        if not self.h:
            raise ValueError("spreading factor should be between 6 and 12")
        self.sps = self.L.lr_sps(self.h)
        self.n_bins = self.L.lr_bins(self.h)
        self.n_bins_hdr = self.L.lr_bins_hdr(self.h)
        self.decim = self.L.lr_decim(self.h)
        self.delay_after_sync = self.L.lr_delay_after_sync(self.h)
        self.output_multiple = self.L.lr_output_multiple(self.h)
        self.bits_per_symbol = self.L.lr_bits_per_symbol(self.h)
        self.dt = self.L.lr_dt(self.h)

    def __del__(self):
        if getattr(self, "h", None):
            self.L.lr_destroy(self.h)
            self.h = None

    def _table(self, name, n, dtype):
        p = getattr(self.L, name)(self.h)
        return np.frombuffer(C.string_at(p, n * np.dtype(dtype).itemsize), dtype=dtype).copy()

    downchirp = property(lambda s: s._table("lr_downchirp", s.sps, np.complex64))
    upchirp = property(lambda s: s._table("lr_upchirp", s.sps, np.complex64))
    downchirp_ifreq = property(lambda s: s._table("lr_downchirp_ifreq", s.sps, np.float32))
    upchirp_ifreq = property(lambda s: s._table("lr_upchirp_ifreq", s.sps, np.float32))
    upchirp_ifreq_v = property(lambda s: s._table("lr_upchirp_ifreq_v", 3 * s.sps, np.float32))

    @staticmethod
    def _iq(x):
        return np.ascontiguousarray(x, dtype=np.complex64)

    def ifreq(self, x):
        x = self._iq(x)
        out = np.empty(x.size, np.float32)
        self.L.lr_instantaneous_frequency(self.h, _ptr(x), _ptr(out), x.size)
        return out

    def get_shift_fft(self, x):
        x = self._iq(x)
        assert x.size >= self.sps
        mag = C.c_float()
        b = self.L.lr_get_shift_fft(self.h, _ptr(x), C.addressof(mag))
        return int(b), float(mag.value)

    def spectrum(self, x):
        x = self._iq(x)
        assert x.size >= self.sps
        out = np.empty(self.n_bins, np.complex64)
        self.L.lr_get_shift_fft_spectrum(self.h, _ptr(x), _ptr(out))
        return out

    def grad_idx(self, x):
        x = self._iq(x)
        assert x.size >= self.sps
        return int(self.L.lr_max_frequency_gradient_idx(self.h, _ptr(x)))

    def fine_sync(self, x, bin_idx, search_space):
        x = self._iq(x)
        assert x.size >= self.sps
        return int(self.L.lr_fine_sync(self.h, _ptr(x), bin_idx, search_space))

    def autocorr(self, x):
        x = self._iq(x)
        assert x.size >= 2 * self.sps
        return float(self.L.lr_detect_preamble_autocorr(self.h, _ptr(x)))

    @property
    def energy_threshold(self):
        return float(self.L.lr_energy_threshold(self.h))

    def detect_upchirp(self, x):
        x = self._iq(x)
        assert x.size >= 2 * self.sps
        idx = C.c_int32(0)
        c = self.L.lr_detect_upchirp(self.h, _ptr(x), C.addressof(idx))
        return float(c), int(idx.value)

    def detect_downchirp(self, x):
        x = self._iq(x)
        assert x.size >= self.sps
        return float(self.L.lr_detect_downchirp(self.h, _ptr(x)))

    def experimental_determine_cfo(self, x):
        x = self._iq(x)
        assert x.size >= self.sps
        return float(self.L.lr_experimental_determine_cfo(self.h, _ptr(x)))

    def energy(self, x):
        x = self._iq(x)
        assert x.size >= self.sps
        return float(self.L.lr_determine_energy(self.h, _ptr(x)))

    def demod_fft_batch(self, iq):
        iq = self._iq(iq)
        n = iq.size // self.sps
        bins = np.empty(n, np.uint32)
        mags = np.empty(n, np.float32)
        self.L.lr_demod_fft_batch(self.h, _ptr(iq), n, _ptr(bins), _ptr(mags))
        return bins, mags

    def demod_grad_batch(self, iq):
        iq = self._iq(iq)
        n = iq.size // self.sps
        bins = np.empty(n, np.uint32)
        self.L.lr_demod_grad_batch(self.h, _ptr(iq), n, _ptr(bins))
        return bins

    def run(self, iq, max_steps=1 << 18):
        iq = self._iq(iq)
        steps = np.zeros(max_steps, STEP_DTYPE)
        n = C.c_size_t(0)
        consumed = self.L.lr_run(self.h, _ptr(iq), iq.size, _ptr(steps), max_steps, C.addressof(n))
        return int(consumed), steps[: min(n.value, max_steps)]

    def work(self, iq):
        iq = self._iq(iq)
        assert iq.size >= 2 * self.sps
        st = Step()
        c = self.L.lr_work(self.h, _ptr(iq), C.addressof(st))
        return int(c), st

    @property
    def state(self):
        return int(self.L.lr_state(self.h))

    def frames(self, clear=True):
        out = []
        for i in range(self.L.lr_frame_count(self.h)):
            out.append(bytes(C.string_at(self.L.lr_frame_data(self.h, i), self.L.lr_frame_len(self.h, i))))
        if clear:
            self.L.lr_frames_clear(self.h)
        return out

    @property
    def stdout(self):
        return self.L.lr_stdout(self.h).decode()

    # integer stage through the reference's member functions
    def deinterleave(self, words, ppm):
        w = np.ascontiguousarray(words, dtype=np.uint32)
        out = np.zeros(ppm, np.uint8)
        self.L.lr_deinterleave_words(self.h, _ptr(w), w.size, ppm, _ptr(out))
        return out

    def decode_codewords(self, codewords, is_header, cr):
        cw = np.ascontiguousarray(codewords, dtype=np.uint8)
        out = np.zeros(1024, np.uint8)
        consumed = C.c_size_t(0)
        n = self.L.lr_decode_codewords(self.h, _ptr(cw), cw.size, int(is_header), cr, _ptr(out), out.size,
                                       C.addressof(consumed))
        return bytes(out[:n]), int(consumed.value)


def rotl(bits, count, size):
    return int(lib().lr_rotl(bits, count, size))


def hamming_encode_soft(nibble):
    return int(lib().lr_hamming_encode_soft(nibble))


def hamming_decode_soft_byte(v):
    return int(lib().lr_hamming_decode_soft_byte(v))
