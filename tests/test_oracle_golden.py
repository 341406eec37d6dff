"""CPU: the oracle against every golden vector the reference offers for this path
(SURVEY.md 8c): README console output, banner numbers, Hamming code book, whitening tables,
and the committed oracle-output fixtures (tests/golden/golden.json)."""
import hashlib
import json
from pathlib import Path

import numpy as np
import pytest

from conftest import FRAME_CASES, case_decoder_args, make_case_iq
from gr_lora_b200 import tx, whitening

GOLD = json.loads((Path(__file__).parent / "golden" / "golden.json").read_text())


def test_fixture_was_checked_against_the_compiled_reference():
    """tests/golden/make_golden.py refuses to write the fixture unless oracle/_ref (the reference's own
    lib/decoder_impl.cc) reproduces every recorded state, consume amount, bin and frame."""
    assert GOLD["pinned_by_reference"] is True
    assert any("decoder_impl.cc" in ln for ln in GOLD["reference_sources_sha256"])


def test_readme_banner_and_frames(oracle):
    """README.md:77-85: banner for SF7 BW125k @1 MS/s and ' 04 90 40 de ad be ef 70 0d' x5."""
    d = oracle.Decoder(sf=7, cr=4, crc=True)
    assert d.stdout == GOLD["readme"]["banner"]
    fs = tx.encode_frame(bytes.fromhex("deadbeef700d"), 7, 4)
    x = tx.channel([tx.modulate_frame(fs, 7)] * 5, sf=7, snr_db=40.0, seed=0x4C6F5201, gap_symbols=97.66)  # ~100 ms gaps
    d.run(x)
    lines = d.stdout[len(GOLD["readme"]["banner"]):].splitlines()
    assert len(lines) == 5
    for ln in lines:
        assert ln.startswith(GOLD["readme"]["line"])
    frames = d.frames()
    assert [f[15:].hex() for f in frames] == ["049040deadbeef700d"] * 5
    assert all(len(f) == 15 + 3 + 6 for f in frames)


def test_header_bytes_match_readme():
    """The 3 header bytes of the README golden are len=4, cr=4, crc=1 + the LoRa header checksum."""
    assert tx.header_bytes(4, 4, 1).hex() == "049040"


def test_hamming_codebook(oracle):
    """hamming_encode_soft code book (include/lora/utilities.h:257-264), SURVEY 8a B4."""
    L = oracle.lib()
    book = [L.lo_hamming84_encode(v) for v in range(16)]
    assert bytes(book).hex() == "00d25587994bcc1ee133b46678aa2dff"
    assert list(tx.HAMMING84) == book
    for v in range(16):
        cw = book[v]
        assert L.lo_hamming84_decode(cw) == v and L.lo_hamming_decode_soft_byte(cw) == v
        for b in range(8):       # every single-bit error is corrected by both decoders
            assert L.lo_hamming84_decode(cw ^ (1 << b)) == v
            assert L.lo_hamming_decode_soft_byte(cw ^ (1 << b)) == v
    # minimum distance 4
    assert min(bin(a ^ b).count("1") for i, a in enumerate(book) for b in book[i + 1:]) == 4


def test_whitening_tables():
    assert len(whitening.PRNG_HEADER) == 13 and not any(whitening.PRNG_HEADER)
    assert len(whitening.PRNG_PAYLOAD_CR56) == 516 and len(whitening.PRNG_PAYLOAD_CR78) == 518
    h = hashlib.sha256()
    for name in ("prng_header", "prng_payload_cr56", "prng_payload_cr78"):
        h.update(name.encode() + b"\0" + getattr(whitening, name.upper()) + b"\0")
    assert h.hexdigest() == whitening.SHA256
    # the same digest taken by tools/gen_tables.py over the reference's lib/tables.h, recorded from that source
    assert (Path(__file__).parent / "golden" / "reference_tables.sha256").read_text().split()[0] == whitening.SHA256


def test_derived_parameters(oracle):
    """A1, lib/decoder_impl.cc:69-91."""
    for sf in range(7, 13):
        d = oracle.Decoder(sf=sf)
        assert d.n_bins == 1 << sf and d.sps == 8 << sf and d.decim == 8
    with pytest.raises(ValueError):
        oracle.Decoder(sf=5)
    with pytest.raises(ValueError):
        oracle.Decoder(sf=14)


def test_fft_vs_gradient_mapping(oracle):
    """SURVEY 8a row A7 probe: on clean aligned symbols grad == (fft - 1) mod N, except shift 0."""
    for sf in (7, 9, 12):
        d = oracle.Decoder(sf=sf)
        n = d.n_bins
        vals = np.unique(np.concatenate([np.arange(1, 20), np.random.default_rng(sf).integers(1, n, 40), [n - 1, n // 2]]))
        x = tx.synth_symbols(vals, sf)
        fb, _ = d.demod_fft_batch(x)
        gb = d.demod_grad_batch(x)
        assert np.array_equal(fb, vals)
        assert np.array_equal(gb, (vals - 1) % n)
        x0 = tx.synth_symbols([0], sf)      # the wrap sits on the window edge: gradient sees nothing
        assert d.get_shift_fft(x0)[0] == 0 and d.grad_idx(x0) == 0


@pytest.mark.parametrize("case", FRAME_CASES, ids=[c[0] for c in FRAME_CASES])
def test_frame_fixtures(oracle, case):
    """TX -> oracle state machine reproduces the committed fixture (frames, consume sequence, bins)."""
    g = GOLD["frames"][case[0]]
    x, fs, payload = make_case_iq(case)
    assert hashlib.sha256(x.tobytes()).hexdigest() == g["iq_sha256"], "synthetic capture is not reproducible"
    assert [int(s) for s in fs.shifts] == g["shifts"]
    d = oracle.Decoder(**case_decoder_args(case))
    consumed, steps = d.run(x)
    assert consumed == g["consumed"]
    assert "".join(str(int(s)) for s in steps["state"]) == g["states"]
    assert [int(c) for c in steps["consumed"]] == g["consumes"]
    assert [int(b) for b in steps["bin"] if b >= 0] == g["bins"]
    assert [f.hex() for f in d.frames()] == g["frames"]
    assert d.stdout == g["stdout"]


@pytest.mark.parametrize("case", [c for c in FRAME_CASES if c[0] not in ("sf7_cr3",)], ids=lambda c: c[0])
def test_frames_decode_to_payload(oracle, case):
    """Round trip: what the TX encoded is what the reference algorithm prints."""
    name, sf, cr, implicit, crc, rr, payload_hex, snr, seed = case
    frames = GOLD["frames"][name]["frames"]
    assert len(frames) == 2
    for f in frames:
        body = bytes.fromhex(f)[18:]
        assert body[:len(bytes.fromhex(payload_hex))].hex() == payload_hex
        if not implicit:
            assert bytes.fromhex(f)[15:18] == tx.header_bytes(len(payload_hex) // 2 - (2 if crc else 0), cr, int(crc))


def test_fft_demod_mode_decodes_where_gradient_cannot(oracle):
    """sf7_cr3 contains a symbol with gradient index N-1 (chirp shift 0): the reference's
    gradient demodulator reads 0 there and cr=3 cannot absorb the extra bit error; the FFT
    demodulator ((fft-1) mod N) gets the payload right."""
    case = [c for c in FRAME_CASES if c[0] == "sf7_cr3"][0]
    x, fs, payload = make_case_iq(case)
    assert 0 in fs.shifts
    d = oracle.Decoder(**case_decoder_args(case), demod=oracle.DEMOD_FFT)
    d.run(x)
    assert [f[18:18 + len(payload)] for f in d.frames()] == [payload] * 2
    g = GOLD["frames"]["sf7_cr3"]["frames"]
    assert all(bytes.fromhex(f)[18:18 + len(payload)] != payload for f in g)


def test_k1_fixtures(oracle):
    for sf in range(7, 13):
        g = GOLD["k1"][str(sf)]
        from golden.make_golden import k1_case
        vals, x = k1_case(sf, g["n"], g["snr_db"], g["seed"])
        assert [int(v) for v in vals] == g["values"]
        d = oracle.Decoder(sf=sf)
        fb, fm = d.demod_fft_batch(x)
        assert [int(b) for b in fb] == g["fft_bins"]
        np.testing.assert_allclose(fm, np.array(g["fft_mags"], np.float32), rtol=2e-5)
        assert [int(b) for b in fb] == g["values"]          # 0 dB in fs bandwidth is easy for the FFT demod


def test_edge_inputs(oracle):
    """Empty / silent / too-short inputs (the reference's work() is never called with < 2*sps)."""
    d = oracle.Decoder(sf=7)
    c, steps = d.run(np.zeros(100, np.complex64))
    assert c == 0 and len(steps) == 0
    c, steps = d.run(np.zeros(8 * 1024, np.complex64))       # all-zero: autocorr is NaN -> stays in DETECT
    assert c == 7 * 1024 and set(steps["state"]) == {0} and not d.frames()
    rng = np.random.default_rng(1)
    noise = (rng.standard_normal(20 * 1024) + 1j * rng.standard_normal(20 * 1024)).astype(np.complex64)
    d.run(noise)
    assert not d.frames()
