import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def have_gpu() -> bool:
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


@pytest.fixture(scope="session")
def oracle():
    from oracle import oracle as O
    O.lib()
    return O


# ---- shared case list: the golden fixtures, the oracle tests and the GPU parity tests all use it
FRAME_CASES = [
    # name, sf, cr, implicit, crc, reduced_rate, payload hex (incl. CRC bytes when crc), snr_db, seed
    ("readme_sf7_cr4", 7, 4, False, True, False, "deadbeef700d", 40.0, 0x4C6F5201),
    ("sf7_cr1", 7, 1, False, True, False, "deadbeef700d", 40.0, 11),
    ("sf7_cr2", 7, 2, False, False, False, "88", 40.0, 12),
    ("sf7_cr3", 7, 3, False, True, False, "ffffffffffffffffffff1234", 40.0, 13),
    ("sf8_cr4", 8, 4, False, True, False, "deadbeefdeadbeefdeadbeefdeadbeefdeadbeef0102", 40.0, 14),
    ("sf8_cr1", 8, 1, False, False, False, "00010203040506070809", 40.0, 15),
    ("sf9_cr2", 9, 2, False, True, False, "deadbeef700d", 40.0, 16),
    ("sf9_cr3", 9, 3, False, False, False, "48656c6c6f204c6f526121", 40.0, 17),
    ("sf10_cr4", 10, 4, False, True, False, "deadbeef700d", 40.0, 18),
    ("sf10_cr1_implicit", 10, 1, True, False, False, "00112233445566778899aabbccddeeff", 40.0, 0x4C6F5205),
    ("sf11_cr4_rr", 11, 4, False, True, True, "deadbeef700d", 40.0, 19),
    ("sf12_cr4_rr", 12, 4, False, True, True, "8899", 40.0, 20),
    ("sf7_cr4_implicit", 7, 4, True, True, False, "cafebabe0102", 40.0, 21),
]


def make_case_iq(case, n_frames=2, cfo_hz=0.0):
    """Deterministic IQ capture for a FRAME_CASES entry (same on every machine)."""
    from gr_lora_b200 import tx
    name, sf, cr, implicit, crc, rr, payload_hex, snr, seed = case
    payload = bytes.fromhex(payload_hex)
    fs = tx.encode_frame(payload, sf, cr, explicit=not implicit, has_crc=crc, reduced_rate=rr)
    # SF11/12: a sync word of 0x12 (shifts 8, 16) looks like a plain upchirp to the reference's
    # Pearson gate (c < -0.97, lib/decoder_impl.cc:801) and derails its timing; use larger shifts.
    frame = tx.modulate_frame(fs, sf, sync_word=0x78 if sf >= 11 else 0x12)
    x = tx.channel([frame] * n_frames, sf=sf, snr_db=snr, seed=seed, cfo_hz=cfo_hz)
    return x, fs, payload


def make_capture(payload, sf, cr, crc, seed, n_frames=1, snr_db=38.0, lead=2.6, sfo_ppm=0.0, cfo_hz=0.0):
    """Synthetic stand-in for one capture of the reference's test suites (apps/generate_test_suites.py:157-203):
    explicit header, reduced rate above SF10, optional sampling-clock offset (ppm) and CFO.  Shared by the GPU parity
    tests and the CPU test that pins the oracle to the compiled reference, so both see the same IQ."""
    from gr_lora_b200 import tx
    fsy = tx.encode_frame(payload, sf, cr, has_crc=crc, reduced_rate=sf > 10)
    frame = tx.modulate_frame(fsy, sf, sync_word=0x78 if sf >= 11 else 0x12)
    x = tx.channel([frame] * n_frames, sf=sf, snr_db=None, seed=seed, lead_symbols=lead, cfo_hz=cfo_hz).astype(np.complex128)
    if sfo_ppm:
        # transmitter clock off by sfo_ppm: resample by linear interpolation (band-limited enough at 8x oversampling)
        t = np.arange(int(x.size / (1 + sfo_ppm * 1e-6))) * (1 + sfo_ppm * 1e-6)
        i0 = np.floor(t).astype(np.int64)
        fr = t - i0
        i1 = np.minimum(i0 + 1, x.size - 1)
        x = x[i0] * (1 - fr) + x[i1] * fr
    x = x + tx.awgn(x.size, snr_db, np.random.default_rng(seed))
    return x.astype(np.complex64)


@pytest.fixture(scope="session")
def ref():
    """The reference's own decoder_impl.cc compiled against stand-in headers (oracle/_ref, oracle/ref.py), answering from
    its recorded outputs (tests/golden/refcalls.py) so that the comparisons run without the reference."""
    from golden.refcalls import open_reference
    r, store = open_reference()
    yield r
    if store.live is not None:
        store.save()


def case_decoder_args(case):
    name, sf, cr, implicit, crc, rr, payload_hex, snr, seed = case
    return dict(samp_rate=1e6, bandwidth=125000, sf=sf, implicit=implicit, cr=cr, crc=crc, reduced_rate=rr,
                disable_drift_correction=False)


def twiddle_table(sps):
    j = np.arange(sps)
    a = -2.0 * np.pi * j / sps
    return (np.cos(a) + 1j * np.sin(a)).astype(np.complex64)
