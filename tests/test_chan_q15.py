"""Complex int16 channelizer (t41rx_chan_create_q15, t41rx_chan_process_device_q15): interleaved (I, Q) int16 pairs at
M x 96 kS/s (M = 64 or 512), as wideband I/Q digitizers stream them (sc16), cut into the complex channelizer's channels.

x = (I + jQ) / 32768 is exact in float32, and the kernel's 2^-15 is folded into the taps (exact too), so the q15
channelizer gives the bits of the float channelizer fed with s / 32768.  The GPU tier checks exactly that, over map
changes, shifts and call splits; every accuracy, tuning and end-to-end property of the float path (test_channelizer.py,
test_chan_tuning.py) then holds for the q15 path as well.

CPU tier: the refusals at creation, the argument clash in Channelizer, synth.wideband_q15.  GPU tier: bit-identity with
the float path, bit-identity across call splits, argument checks.
"""
import ctypes as C

import numpy as np
import pytest

from chan_driver import channelize
from t41_sdr_b200 import rx, synth

CHANNELS = (64, 512)
BLOCK = rx.BLOCK
EINVAL, ENODEV = -1, -4
FILL = 12345.0


# ---------------------------------------------------------------- CPU tier

def test_create_q15_checks_its_arguments():
    h = C.c_void_p()
    for m in (128, 1024, 256, 100):
        assert rx.lib().t41rx_chan_create_q15(C.byref(h), m, 4, 0) == EINVAL
        assert b"t41rx_chan_create_q15" in rx.lib().t41rx_last_error()
    for n_recv in (0, -1):
        assert rx.lib().t41rx_chan_create_q15(C.byref(h), 64, n_recv, 0) == EINVAL
    assert not h.value


def test_create_q15_without_device_is_enodev():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    h = C.c_void_p()
    assert rx.lib().t41rx_chan_create_q15(C.byref(h), 512, 4, 0) == ENODEV
    assert b"no CUDA device" in rx.lib().t41rx_last_error()
    assert not h.value


def test_real_and_q15_together_are_refused():
    with pytest.raises(ValueError):
        rx.Channelizer(64, 4, real=True, q15=True)


def test_wideband_q15_is_the_quantised_wideband_sum():
    M, T = 64, 2
    sig = [("tone", 1.1e6, {"amp": 0.3}), ("am", -0.4e6, {"amp": 0.2}), ("nfm", 2.5e6, {"amp": 0.1})]
    s = synth.wideband_q15(4, M, T, sig, sigma=0.05, start_block=3)
    assert s.dtype == np.int16 and s.shape == (T * BLOCK * M // 2, 2)
    z = synth._wideband_sum(4, M, T, sig, 0.05, 3)
    assert np.array_equal(s[:, 0], np.clip(np.round(32768.0 * z.real), -32768, 32767))
    assert np.array_equal(s[:, 1], np.clip(np.round(32768.0 * z.imag), -32768, 32767))
    # wideband() is the same sum rounded to float32: within one step of it
    f = synth.wideband(4, M, T, sig, sigma=0.05, start_block=3)
    assert np.abs(s.astype(np.float64) - 32768.0 * f.astype(np.float64)).max() <= 0.5 + 1e-3
    # saturation: a tone at 1.5 x full scale clips at both ends of both components
    loud = synth.wideband_q15(0, M, 1, [("tone", 96000.0, {"amp": 1.5})])
    for c in (0, 1):
        assert loud[:, c].max() == 32767 and loud[:, c].min() == -32768
    z = synth._wideband_sum(0, M, 1, [("tone", 96000.0, {"amp": 1.5})], 0.0, 0)
    assert np.all(loud[32768.0 * z.real >= 32767.5, 0] == 32767)
    assert np.all(loud[32768.0 * z.real <= -32768.5, 0] == -32768)


# ---------------------------------------------------------------- GPU tier

def _test_capture(M, n_blocks, seed):
    """a seeded wideband_q15 capture with full-scale samples (-32768 and 32767, in I and in Q) scattered through it"""
    r = np.random.default_rng(seed)
    half = synth.wideband_rate(M) / 2
    sig = [("tone", float(r.uniform(-half, half)), {"amp": float(r.uniform(0.03, 0.15))}) for _ in range(6)]
    sig.append(("tone", rx.chan_centre(M, M // 2) + 1234.5, {"amp": 0.1}))
    s = synth.wideband_q15(seed, M, n_blocks, sig, sigma=0.05)
    for value in (-32768, 32767):
        idx = r.choice(s.shape[0], 64, replace=False)
        s[idx, r.integers(0, 2, idx.size)] = value
        s[r.choice(s.shape[0], 8, replace=False)] = value
    return s


@pytest.mark.gpu
@pytest.mark.parametrize("M", CHANNELS)
def test_q15_is_bit_identical_to_float_on_s_over_32768(M):
    """A q15 channelizer on s and a float channelizer on s / 32768 (exact) run the same schedule: calls of 1 + 2 + 5
    blocks, a map change before the third call (receivers unmapped and remapped), shifts set before the first and the
    second call (positive, negative, +-96000, +-191999, two shifts on one channel), receivers 7 ... 9 never shifted.
    Every iq value is bit-identical; rows of unmapped receivers keep their fill."""
    capture = _test_capture(M, 8, 40 + M)
    assert (capture == -32768).any() and (capture == 32767).any()
    map1 = [0, 1, M // 2 - 1, M // 2, M - 1, 5, 5, -1, 3, 7]
    map2 = [5, -1, 0, M - 1, M // 2, 5, 3, 2, -1, 7]
    shifts1 = [12345, -54321, 96000, -96000, 0, 777, -191999]
    shifts2 = [191999, -191999, 4000, 0]
    calls, maps, shifts = [1, 2, 5], [map1, None, map2], [shifts1, shifts2, None]
    got = channelize(M, len(map1), capture, calls, maps, shifts, q15=True)
    want = channelize(M, len(map1), capture.astype(np.float32) / 32768.0, calls, maps, shifts, q15=False)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    assert np.all(got[7, :3] == FILL)
    assert np.all(got[1, 3:] == FILL) and np.all(got[8, 3:] == FILL)
    for r in (0, 2, 3, 4, 5, 6, 9):
        assert not np.any(got[r] == FILL), r


@pytest.mark.gpu
@pytest.mark.parametrize("M", CHANNELS)
def test_split_calls_are_bit_identical_q15(M):
    """The same q15 capture in one 8-block call and in 1 + 2 + 5 blocks gives the same bits, with and without shifts."""
    capture = _test_capture(M, 8, 7)
    chmap = [3, 40 % M, -1, 3, M // 2, 0]
    for sh in (None, [48000, -20000, 0, 0, 95999, -191999]):
        one = channelize(M, 6, capture, [8], [chmap], [sh], q15=True)
        split = channelize(M, 6, capture, [1, 2, 5], [chmap, None, None], [sh, None, None], q15=True)
        assert np.array_equal(one.view(np.uint32), split.view(np.uint32))
        assert np.all(one[2] == FILL)


@pytest.mark.gpu
def test_argument_checks_q15():
    import torch
    M = 64
    per_block = BLOCK * M // 2
    cap = torch.zeros((per_block + 8, 2), dtype=torch.int16, device="cuda")
    cap_f = torch.zeros((per_block, 2), dtype=torch.float32, device="cuda")
    iq = torch.zeros(2 * BLOCK * 2 + 2, dtype=torch.float32, device="cuda")    # 2 receivers x 1 block, and room to offset
    L = rx.lib()
    with rx.Channelizer(M, 2, q15=True) as ch:
        ch.set_map([M - 1, 0])
        with pytest.raises(rx.T41RxError, match="channel out of range"):
            ch.set_map([M, 0])
        for off in (4, 8):               # 4- and 8-byte aligned, not 16
            with pytest.raises(rx.T41RxError, match="aligned"):
                ch.process_device(cap.data_ptr() + off, iq.data_ptr(), 1)
        with pytest.raises(rx.T41RxError, match="aligned"):
            ch.process_device(cap.data_ptr(), iq.data_ptr() + 4, 1)
        for nb in (0, -1):
            assert L.t41rx_chan_process_device_q15(ch._h, cap.data_ptr(), iq.data_ptr(), nb, None) == EINVAL
        assert L.t41rx_chan_process_device_q15(ch._h, None, iq.data_ptr(), 1, None) == EINVAL
        assert L.t41rx_chan_process_device_q15(ch._h, cap.data_ptr(), None, 1, None) == EINVAL
        assert L.t41rx_chan_process_device_q15(None, cap.data_ptr(), iq.data_ptr(), 1, None) == EINVAL
        # the other kinds' process calls
        assert L.t41rx_chan_process_device(ch._h, cap_f.data_ptr(), iq.data_ptr(), 1, None) == EINVAL
        assert b"t41rx_chan_process_device_q15" in L.t41rx_last_error()
        assert L.t41rx_chan_process_device_real(ch._h, cap.data_ptr(), iq.data_ptr(), 1, None) == EINVAL
        assert b"t41rx_chan_process_device_q15" in L.t41rx_last_error()
        ch.process_device(cap.data_ptr(), iq.data_ptr(), 1)
        ch.synchronize()
    with rx.Channelizer(M, 2) as ch:
        ch.set_map([0, 1])
        assert L.t41rx_chan_process_device_q15(ch._h, cap.data_ptr(), iq.data_ptr(), 1, None) == EINVAL
    with rx.Channelizer(128, 2, real=True) as ch:
        ch.set_map([0, 1])
        assert L.t41rx_chan_process_device_q15(ch._h, cap.data_ptr(), iq.data_ptr(), 1, None) == EINVAL
        assert b"t41rx_chan_process_device_real" in L.t41rx_last_error()
