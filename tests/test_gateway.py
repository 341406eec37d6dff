"""CPU: the gateway receiver's C ABI (lora_b200_gateway_*): record layouts, argument checks that run before any device is
looked for, the no-GPU failure, and the gather's index map and tail bookkeeping run on the host (build/host_emul.so)."""
import ctypes as C

import numpy as np
import pytest

from conftest import have_gpu
import gr_lora_b200
from gr_lora_b200 import _native as N, build as B
from gr_lora_b200.gateway import FRAME_DTYPE


def test_config_and_frame_records_match_the_header():
    G = N.GatewayConfig
    assert C.sizeof(G) == 56
    offs = {"samp_rate": 0, "center_freq": 4, "channel_list": 8, "n_channels": 16, "bandwidth": 20, "decimation": 24, "sf_mask": 28,
            "reduced_rate_mask": 32, "implicit": 36, "cr": 37, "crc": 38, "demod": 39, "conj": 40, "disable_drift_correction": 41,
            "reserved": 42, "device": 44, "max_in_per_call": 48, "max_frames_per_call": 52}
    assert {n: getattr(G, n).offset for n in offs} == offs
    # lora_b200_gateway_frame = channel | sf | lora_b200_frame (584 bytes)
    assert gr_lora_b200.decoder.FRAME_DTYPE.itemsize == 584
    assert FRAME_DTYPE.itemsize == 592
    assert FRAME_DTYPE.fields["channel"][1] == 0 and FRAME_DTYPE.fields["sf"][1] == 4 and FRAME_DTYPE.fields["stream"][1] == 8
    assert FRAME_DTYPE.fields["bytes"][1] == 8 + 20


def _cfg(**kw):
    cl = (C.c_float * 2)(868.1e6, 868.3e6)
    base = dict(samp_rate=4e6, center_freq=868.2e6, channel_list=C.cast(cl, C.POINTER(C.c_float)), n_channels=2, bandwidth=125000,
                decimation=4, sf_mask=(1 << 7) | (1 << 9), cr=4, crc=1, device=-1)
    base.update(kw)
    return N.GatewayConfig(**base), cl


@pytest.mark.parametrize("bad,match", [
    (dict(n_channels=0), "empty channel list"),
    (dict(channel_list=None), "empty channel list"),
    (dict(decimation=0), "decimation"),
    (dict(sf_mask=0), "sf_mask"),
    (dict(sf_mask=1 << 6), "sf_mask"),
    (dict(sf_mask=(1 << 7) | (1 << 13)), "sf_mask"),
    (dict(cr=5), "coding rate"),
    (dict(reduced_rate_mask=1 << 3), "reduced_rate_mask"),
])
def test_invalid_arguments_are_rejected_before_the_device_check(bad, match):
    L = N.lib()
    cfg, _keep = _cfg(**bad)
    assert not L.lora_b200_gateway_create(C.byref(cfg))
    msg = L.lora_b200_last_error().decode()
    assert match in msg and "no CUDA device" not in msg


def test_null_handles_are_rejected():
    L = N.lib()
    nf = C.c_size_t(0)
    assert L.lora_b200_gateway_work(None, None, 0, 1, C.byref(nf)) == N.EINVAL
    assert L.lora_b200_gateway_reset(None) == N.EINVAL
    c, p = C.c_uint64(0), C.c_uint32(0)
    assert L.lora_b200_gateway_position(None, 0, 7, C.byref(c), C.byref(p)) == N.EINVAL
    L.lora_b200_gateway_destroy(None)


def test_python_arguments_reach_the_checks():
    with pytest.raises(RuntimeError, match="sf_mask"):
        gr_lora_b200.gateway(4e6, 868e6, [868.1e6], 125000, sfs=(6,))
    with pytest.raises(RuntimeError, match="empty channel list"):
        gr_lora_b200.gateway(4e6, 868e6, [], 125000)


@pytest.mark.skipif(have_gpu(), reason="checks the no-GPU failure mode")
def test_no_cpu_fallback():
    with pytest.raises(RuntimeError, match="no CUDA device"):
        gr_lora_b200.gateway(4e6, 868e6, [868.1e6, 868.3e6], 125000, decimation=4)


@pytest.fixture(scope="module")
def emul():
    L = C.CDLL(str(B.build_host_emul()))
    L.lb_emul_gw_gather.restype = C.c_int64
    L.lb_emul_gw_gather.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p]
    L.lb_emul_gw_pending.restype = C.c_uint32
    L.lb_emul_gw_pending.argtypes = [C.c_uint32, C.c_uint32]
    return L


@pytest.mark.parametrize("seed", range(4))
def test_gather_index_map_and_bookkeeping(emul, seed):
    """One stream over many calls with random consumption: every call presents exactly the stream's unconsumed items
    followed by the new chunk (pending' = pending - consumed + M), and an overflow is reported without writing."""
    rng = np.random.default_rng(seed)
    cap, sps = 4096 + 2 * 256 + 256, 256
    stream = (rng.standard_normal(200000) + 1j * rng.standard_normal(200000)).astype(np.complex64)
    bufs = [np.zeros(cap, np.complex64), np.zeros(cap, np.complex64)]
    cur, read, fed, pending, off, length = 0, 0, 0, 0, 0, 0
    for _ in range(200):
        m = int(rng.integers(0, 4097))
        o = stream[fed:fed + m].copy()
        m = o.size
        nxt = bufs[cur ^ 1]
        n = emul.lb_emul_gw_gather(bufs[cur].ctypes.data, off, pending, o.ctypes.data, m, cap, nxt.ctypes.data)
        assert n == pending + m
        fed += m
        assert np.array_equal(nxt[:n], stream[read:read + n])         # the tail from its offset, then the new items
        cur ^= 1
        length = n
        # the state machine consumes in steps and stops when fewer than 2 sps items are left
        consumed = 0
        while length - consumed >= 2 * sps:
            consumed += int(rng.integers(1, sps + sps // 4 + 1))
        consumed = min(consumed, length)
        off = consumed
        pending = emul.lb_emul_gw_pending(length, consumed)
        assert pending == length - consumed and pending < 2 * sps
        read += consumed
    # a stream that stopped early (max_frames_per_call) keeps a long tail: a chunk that does not fit is refused untouched
    big = np.full(cap, 7 + 7j, np.complex64)
    o = np.zeros(cap, np.complex64)
    dst = np.full(cap, 1 + 1j, np.complex64)
    assert emul.lb_emul_gw_gather(big.ctypes.data, 0, cap - 100, o.ctypes.data, 101, cap, dst.ctypes.data) == -1
    assert np.all(dst == 1 + 1j)
    assert emul.lb_emul_gw_gather(big.ctypes.data, 0, cap - 100, o.ctypes.data, 100, cap, dst.ctypes.data) == cap
    assert emul.lb_emul_gw_pending(10, 12) == 0
