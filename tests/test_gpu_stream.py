"""GPU parity: the whole receive path (state machine kernel + K8) through the C ABI's work() against
the oracle's restatement of decoder_impl::work and the committed fixtures."""
import json
from pathlib import Path

import numpy as np
import pytest

from conftest import FRAME_CASES, case_decoder_args, make_case_iq

pytestmark = pytest.mark.gpu
GOLD = json.loads((Path(__file__).parent / "golden" / "golden.json").read_text())


@pytest.fixture(scope="module")
def torch():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no GPU")
    return torch


def gpu_decoder(case, **kw):
    import gr_lora_b200 as G
    a = case_decoder_args(case)
    return G.decoder(a["samp_rate"], a["bandwidth"], a["sf"], a["implicit"], a["cr"], a["crc"], a["reduced_rate"],
                     a["disable_drift_correction"], quiet=True, **kw)


@pytest.mark.parametrize("case", FRAME_CASES, ids=[c[0] for c in FRAME_CASES])
def test_frames_bit_exact_and_trace_equal(torch, case):
    """Gradient demodulator (the reference's live path): frames bit-exact, and the per-step
    (state, consume, bin) trace equal to the oracle's."""
    g = GOLD["frames"][case[0]]
    x, fs, payload = make_case_iq(case)
    dec = gpu_decoder(case, trace_capacity=4096, max_items_per_call=x.size)
    consumed = dec.work(x)
    assert [f.hex() for _, f in dec.frames] == g["frames"]
    assert consumed == g["consumed"]
    tr = dec.trace()
    assert "".join(str(s[0]) for s in tr) == g["states"]
    assert [s[1] for s in tr] == g["consumes"]
    assert [s[2] for s in tr if s[2] >= 0] == g["bins"]
    dec.close()


@pytest.mark.parametrize("case", FRAME_CASES, ids=[c[0] for c in FRAME_CASES])
def test_fft_demod_decodes_transmitted_payload(torch, case):
    """North-star demodulator (dechirp+FFT+argmax, bin-1 mapping): decoded bytes equal what was sent."""
    name, sf, cr, implicit, crc, rr, payload_hex, snr, seed = case
    x, fs, payload = make_case_iq(case)
    dec = gpu_decoder(case, demod="fft", max_items_per_call=x.size)
    dec.work(x)
    got = [f[18:18 + len(payload)] for _, f in dec.frames]
    assert got == [payload] * 2
    if name != "sf7_cr3":        # where the gradient path is right too, the two paths publish identical frames
        assert [f.hex() for _, f in dec.frames] == GOLD["frames"][name]["frames"]
    dec.close()


def test_fft_mode_matches_oracle_fft_mode(torch, oracle):
    for name in ("readme_sf7_cr4", "sf9_cr2", "sf11_cr4_rr"):
        case = [c for c in FRAME_CASES if c[0] == name][0]
        x, fs, payload = make_case_iq(case)
        od = oracle.Decoder(**case_decoder_args(case), demod=oracle.DEMOD_FFT)
        oc, osteps = od.run(x)
        dec = gpu_decoder(case, demod="fft", trace_capacity=4096, max_items_per_call=x.size)
        c = dec.work(x)
        assert c == oc
        assert [f for _, f in dec.frames] == od.frames()
        tr = dec.trace()
        assert [s[1] for s in tr] == [int(v) for v in osteps["consumed"]]
        assert [s[2] for s in tr] == [int(v) for v in osteps["bin"]]
        dec.close()


def test_readme_stdout(torch, capsys):
    """Banner + hex lines exactly as the reference prints them (README.md:77-85)."""
    import gr_lora_b200 as G
    from gr_lora_b200 import tx
    fs = tx.encode_frame(bytes.fromhex("deadbeef700d"), 7, 4)
    x = tx.channel([tx.modulate_frame(fs, 7)] * 5, sf=7, snr_db=40.0, seed=0x4C6F5201, gap_symbols=97.66)
    rx = G.lora_receiver(1e6, 868.1e6, [868.1e6], 125000, 7, False, 4, True, max_items_per_call=1 << 19)
    rx.run(x)
    out = capsys.readouterr().out
    assert out.startswith(GOLD["readme"]["banner"])
    lines = out[len(GOLD["readme"]["banner"]):].splitlines()
    assert len(lines) == 5 and all(ln.startswith(GOLD["readme"]["line"]) for ln in lines)
    assert len(rx.frames) == 5


@pytest.mark.parametrize("chunk_syms", [2.5, 7, 40])
def test_chunked_feeding_equals_one_shot(torch, chunk_syms):
    """work() called the GNU Radio way: small buffers, caller drops what was consumed and
    re-presents the tail.  Same frames, same total consumption, never reads past n_items."""
    case = FRAME_CASES[0]
    x, fs, payload = make_case_iq(case)
    chunk = int(chunk_syms * 1024)
    dec = gpu_decoder(case, max_items_per_call=chunk)
    total = dec.run(x, chunk_items=chunk)
    g = GOLD["frames"][case[0]]
    assert [f.hex() for _, f in dec.frames] == g["frames"]
    assert total == g["consumed"]
    dec.close()


def test_multi_stream_batch(torch, oracle):
    """n_streams independent streams in one launch (host and device inputs); each stream must
    publish exactly what the oracle publishes for its capture."""
    import gr_lora_b200 as G
    from gr_lora_b200 import tx
    sf, cr, ns = 8, 4, 12
    caps, want = [], []
    for s in range(ns):
        payload = bytes([(s * 17 + k) & 0xFF for k in range(3 + s)])
        fsy = tx.encode_frame(payload, sf, cr, has_crc=False)
        caps.append(tx.channel([tx.modulate_frame(fsy, sf)] * (1 + s % 3), sf=sf, snr_db=38.0, seed=900 + s,
                               lead_symbols=2 + 0.37 * s))
    n = max(c.size for c in caps)
    batch = np.zeros((ns, n), np.complex64)
    for s, c in enumerate(caps):
        batch[s, :c.size] = c
        od = oracle.Decoder(sf=sf, cr=cr, crc=False)
        od.run(batch[s])
        want.append(od.frames())
    for mode in ("host", "device"):
        dec = G.decoder(1e6, 125000, sf, False, cr, False, n_streams=ns, quiet=True, max_items_per_call=n)
        if mode == "host":
            dec.work_batch(batch)
        else:
            t = torch.from_numpy(batch).cuda()
            dec.work_batch(t, n_items=n, stride_items=n, host=0)
        got = [[f for st, f in dec.frames if st == s] for s in range(ns)]
        assert got == want
        dec.close()


def test_noise_and_silence_publish_nothing(torch):
    import gr_lora_b200 as G
    rng = np.random.default_rng(3)
    x = (rng.standard_normal(40 * 1024) + 1j * rng.standard_normal(40 * 1024)).astype(np.complex64)
    dec = G.decoder(1e6, 125000, 7, False, 4, True, quiet=True)
    assert dec.work(x) == 39 * 1024 and not dec.frames and dec.state() == 0     # last start = n - 2*sps
    assert dec.work(np.zeros(10 * 1024, np.complex64)) == 9 * 1024 and not dec.frames
    assert dec.work(np.zeros(100, np.complex64)) == 0         # < 2*sps: nothing to do (output_multiple)
    dec.close()


def test_set_sf_is_refused_like_the_reference(torch, capsys):
    import gr_lora_b200 as G
    dec = G.decoder(1e6, 125000, 7, False, 4, True, quiet=True)
    dec.set_sf(9)
    dec.set_samp_rate(2e6)
    err = capsys.readouterr().err
    assert "Setting the spreading factor during execution is currently not supported" in err
    assert "Setting the sample rate during execution is currently not supported" in err and dec.sps == 1024
    dec.close()


@pytest.mark.parametrize("fs", [500e3, 2e6])
def test_other_sample_rates_gradient_path(torch, oracle, fs):
    """samp_rate / bandwidth != 8 (decimation 4 and 16): the gradient path is generic in sps
    (lib/decoder_impl.cc:83-87); the FFT demodulator is refused there instead of silently falling back."""
    import gr_lora_b200 as G
    from gr_lora_b200 import tx
    sf, cr = 7, 4
    payload = bytes.fromhex("0badc0de1234")
    fsy = tx.encode_frame(payload, sf, cr)
    frame = tx.modulate_frame(fsy, sf, fs=fs)
    x = tx.channel([frame] * 2, sf=sf, fs=fs, snr_db=40.0, seed=3)
    od = oracle.Decoder(samp_rate=fs, sf=sf, cr=cr, crc=True)
    oc, _ = od.run(x)
    want = od.frames()
    assert [f[18:24] for f in want] == [payload] * 2
    dec = G.decoder(fs, 125000, sf, False, cr, True, quiet=True, max_items_per_call=x.size)
    assert dec.sps == int(fs / 125e3) * 128 and dec.decim == int(fs / 125e3)
    assert dec.work(x) == oc and [f for _, f in dec.frames] == want
    dec.close()
    with pytest.raises(RuntimeError, match="samp_rate/bandwidth == 8"):
        G.decoder(fs, 125000, sf, False, cr, True, quiet=True, demod="fft")


@pytest.mark.parametrize("cfo_hz", [0.0, 800.0, -2500.0])
def test_cfo_estimate_equals_reference_function(torch, oracle, ref, cfo_hz):
    """N4: lora_b200_set_cfo_estimate -> experimental_determine_cfo (lib/decoder_impl.cc:730-738) at the SYNC step, on the
    window the reference's commented-out call site would pass (&input[i], :774).  Compared with the reference's own
    function (oracle/_ref, its recorded answers: tests/golden/refcalls.py); frames and the step trace are untouched by the
    option."""
    import gr_lora_b200 as G
    from conftest import make_capture
    x = make_capture(bytes.fromhex("0123456789abcdef"), 8, 4, True, seed=33, cfo_hz=cfo_hz)
    plain = G.decoder(1e6, 125000, 8, False, 4, True, quiet=True, max_items_per_call=x.size, trace_capacity=4096)
    plain.work(x)
    dec = G.decoder(1e6, 125000, 8, False, 4, True, quiet=True, max_items_per_call=x.size, trace_capacity=4096)
    dec.set_cfo_estimate(True)
    dec.work(x)
    assert dec.frames == plain.frames and dec.trace() == plain.trace()
    assert plain.last_cfo() == (0.0, 0)
    cfo, n = dec.last_cfo()
    tr = dec.trace()
    sync_steps = [k for k, s in enumerate(tr) if s[0] == 1]
    assert n == len(sync_steps) >= 1
    k = sync_steps[-1]
    pos = sum(s[1] for s in tr[:k]) + tr[k][1]              # &input[i]: the window start after the SYNC step's consume
    want = ref.RefDecoder(sf=8).experimental_determine_cfo(x[pos:pos + 2048])
    assert abs(cfo - want) < 0.5, (cfo, want)
    # what the number means: a chirp cannot tell a frequency offset from a time shift (61 Hz per sample at SF8) and the window
    # starts where the SYNC correlator put it, so the value is CFO + 61 Hz x (residual misalignment in samples): the
    # reference marks the function experimental and leaves its call commented out.  The claim here is only that the
    # device computes the reference's number.
    dec.close(); plain.close()
