"""GPU: the gateway receiver (lora_b200_gateway_*) on a wideband capture with four channels and four SFs.  The core check is
equivalence: every (channel, SF) stream decodes byte for byte what a standalone channelizer fed the same chunks followed by
a single-stream decoder on that channel decodes, and consumes as much."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

FS_IN, DECIM, CENTER = 4e6, 4, 868.0e6
OFFSETS = (-1.2e6, -0.4e6, 0.4e6, 1.2e6)
SFS = (7, 8, 9, 12)
MAX_IN = 1 << 23


@pytest.fixture(scope="module")
def torch():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no GPU")
    return torch


def _payload(ch, sf, k):
    return bytes([0xA0 + ch, sf, k, 0x5A ^ (16 * ch + sf + k), 0x70, 0x0D])


def _channel_signal(ch):
    """One channel at the decoders' 1 MS/s: one frame of every SF (SF7 twice) back to back, in an order that differs per
    channel so that frames of different SFs overlap across channels.  SF12 is reduced rate (the gateway's default)."""
    from gr_lora_b200 import tx
    order = list(SFS[ch % len(SFS):] + SFS[:ch % len(SFS)])
    parts, sent = [], []
    for sf in order:
        for k in range(2 if sf == 7 else 1):
            p = _payload(ch, sf, k)
            fsy = tx.encode_frame(p, sf, 4, reduced_rate=sf >= 11)
            frame = tx.modulate_frame(fsy, sf, sync_word=0x78 if sf >= 11 else 0x12)
            parts.append(tx.channel([frame], sf=sf, snr_db=None, lead_symbols=3, tail_symbols=4).astype(np.complex128))
            sent.append((sf, p))
    return np.concatenate(parts), sent


@pytest.fixture(scope="module")
def capture():
    """The wideband capture: every channel upsampled to 4 MS/s, shifted to its offset, summed, +15 dB AWGN (as
    test_receiver_with_channelizer_decodes_offset_channel)."""
    from scipy.signal import resample_poly
    from gr_lora_b200 import tx
    sigs, sent = zip(*(_channel_signal(ch) for ch in range(len(OFFSETS))))
    n = max(s.size for s in sigs) * DECIM + 40000
    x = np.zeros(n, np.complex128)
    t = np.arange(n)
    for s, f in zip(sigs, OFFSETS):
        up = resample_poly(s, DECIM, 1)
        x[:up.size] += up * np.exp(2j * np.pi * f * t[:up.size] / FS_IN)
    x += tx.awgn(n, 15.0, np.random.default_rng(17))
    n -= n % DECIM
    return x[:n].astype(np.complex64), sent


def _gateway(conj=False, **kw):
    import gr_lora_b200 as G
    offs = [-f for f in OFFSETS] if conj else list(OFFSETS)
    return G.gateway(FS_IN, CENTER, [CENTER + f for f in offs], 125000, sfs=SFS, decimation=DECIM, conj=conj, max_in_per_call=MAX_IN, **kw)


def _by_stream(frames):
    out = {}
    for r in frames:
        out.setdefault((int(r["channel"]), int(r["sf"])), []).append(bytes(r["bytes"][:r["len"]]))
    return out


def _chunks(n, sizes):
    """chunk boundaries: the given sizes, then 2^20 items at a time"""
    pos, out = 0, []
    for s in sizes:
        out.append((pos, pos + s))
        pos += s
    while pos < n:
        out.append((pos, min(pos + (1 << 20), n)))
        pos = out[-1][1]
    return out


IRREGULAR = [4 * 100, 4 * 123457, 4 * 7, 4 * 654321, 4 * 99999]    # 400 items: shorter than the 962-sample filter history


@pytest.fixture(scope="module")
def standalone(torch, capture):
    """Reference path: the same irregular chunks through a standalone channelizer, then one decoder(n_streams=1) per
    (channel, SF) over that channel's whole output."""
    import gr_lora_b200 as G
    x, _ = capture
    ch = G.channelizer(FS_IN, CENTER, [CENTER + f for f in OFFSETS], 125000, DECIM)
    outs = []
    for a, b in _chunks(x.size, IRREGULAR):
        d_in = torch.from_numpy(x[a:b].copy()).cuda()
        m = (b - a) // DECIM
        d_out = torch.zeros((len(OFFSETS), m), dtype=torch.complex64, device="cuda")
        assert ch.work_dev(d_in, b - a, d_out, m) == m
        outs.append(d_out.cpu().numpy())
    y = np.concatenate(outs, axis=1)
    ch.close()
    frames, consumed = {}, {}
    for c in range(len(OFFSETS)):
        for sf in SFS:
            dec = G.decoder(FS_IN / DECIM, 125000, sf, False, 4, True, reduced_rate=sf >= 11, quiet=True)
            consumed[(c, sf)] = dec.run(y[c])
            frames[(c, sf)] = [f for _, f in dec.frames]
            dec.close()
    return frames, consumed


@pytest.fixture(scope="module")
def irregular_run(torch, capture):
    x, _ = capture
    gw = _gateway()
    frames = np.concatenate([gw.work(x[a:b]) for a, b in _chunks(x.size, IRREGULAR)])
    pos = {(c, sf): gw.position(c, sf) for c in range(len(OFFSETS)) for sf in SFS}
    return gw, frames, pos


def test_every_stream_equals_channelizer_then_decoder(standalone, irregular_run):
    ref_frames, ref_consumed = standalone
    _, frames, pos = irregular_run
    got = _by_stream(frames)
    for key, want in ref_frames.items():
        assert got.get(key, []) == want, key
    assert set(got) <= set(ref_frames)
    for key, (consumed, pending) in pos.items():
        assert consumed == ref_consumed[key], key
        assert pending < 2 * (8 << key[1])


def test_frame_order_is_sf_channel_seq(irregular_run):
    _, frames, _ = irregular_run
    assert np.array_equal(frames["stream"], frames["channel"])
    # within every call the order is (sf, channel, seq); seq grows per stream over the calls
    last = {}
    for r in frames:
        k = (int(r["channel"]), int(r["sf"]))
        assert int(r["seq"]) == last.get(k, -1) + 1
        last[k] = int(r["seq"])


def test_every_payload_is_decoded_on_its_own_stream(capture, irregular_run):
    _, sent = capture
    _, frames, _ = irregular_run
    got = _by_stream(frames)
    for c, lst in enumerate(sent):
        for sf, p in lst:
            assert any(f[18:] == p for f in got.get((c, sf), [])), (c, sf, p.hex())


def test_chunking_does_not_change_the_frames(capture, irregular_run):
    x, _ = capture
    _, frames, _ = irregular_run
    want = _by_stream(frames)
    whole = _gateway()
    assert x.size <= MAX_IN
    assert _by_stream(whole.work(x)) == want
    whole.close()
    regular = _gateway()
    assert _by_stream(regular.run(x, chunk_items=1 << 20)) == want
    # the same gateway after reset(), fed again: the same frames
    regular.reset()
    assert _by_stream(regular.run(x, chunk_items=1 << 20)) == want
    assert regular.position(0, 7)[0] > 0
    regular.close()


def test_device_input_equals_host_input(torch, capture, irregular_run):
    x, _ = capture
    _, frames, _ = irregular_run
    gw = _gateway()
    d = torch.from_numpy(x).cuda()
    got = np.concatenate([gw.work(d[a:b]) for a, b in _chunks(x.size, IRREGULAR)])
    assert _by_stream(got) == _by_stream(frames)
    gw.close()


def test_conjugated_capture_with_mirrored_channels(capture, irregular_run):
    x, _ = capture
    _, frames, _ = irregular_run
    gw = _gateway(conj=True)
    got = gw.run(np.conj(x), chunk_items=1 << 20)
    assert _by_stream(got) == _by_stream(frames)
    gw.close()


def test_bad_chunk_lengths_are_rejected(torch):
    from gr_lora_b200 import _native as N
    gw = _gateway()
    with pytest.raises(N.LoraB200Error, match="multiple of the decimation") as e:
        gw.work(np.zeros(4 * 1000 + 2, np.complex64))
    assert e.value.code == N.EINVAL
    with pytest.raises(N.LoraB200Error, match="max_in_per_call") as e:
        gw.work(np.zeros(MAX_IN + DECIM, np.complex64))
    assert e.value.code == N.EINVAL
    with pytest.raises(N.LoraB200Error, match="not decoded"):
        gw.position(0, 10)
    gw.close()
