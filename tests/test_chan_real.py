"""Real-sampled channelizer (t41rx_chan_create_real, t41rx_chan_process_device_real): an int16 real capture at
M x 96 kS/s (M = 128 or 1024), as a direct-sampling ADC delivers it, cut into channels 0 ... M/2 of 192 kS/s.

CPU tier: the prototype at M = 128 and 1024, where t41rx_chan_tune_real / t41rx_chan_place_real put a receiver and what
they reject, the refusals at creation.  GPU tier: the kernel against the float64 defining formula on x = s / 32768,
bit-identity across call splits and map changes, gain and rejection of a real tone, argument checks, and the chain end
to end on receivers placed by chan_place_real.
"""
import ctypes as C

import numpy as np
import pytest

import cases
import oracle_py as O
from chan_driver import chain, channelize, error_ratio, reference_channel, response_db, rotate
from t41_sdr_b200 import rx, synth

CHANNELS = (128, 1024)
MIRRORED = (rx.DEMOD_USB, rx.DEMOD_LSB, rx.DEMOD_AM, rx.DEMOD_SAM)
PLAIN = (rx.DEMOD_NFM, rx.DEMOD_PSK31)
BLOCK = rx.BLOCK
EINVAL, ENODEV = -1, -4


# ---------------------------------------------------------------- CPU tier

@pytest.mark.parametrize("M", CHANNELS)
def test_prototype_design_real(M):
    taps = rx.chan_taps(M)
    assert taps.dtype == np.float32 and taps.size == 10 * M
    assert np.array_equal(taps, taps[::-1])
    assert abs(float(np.sum(taps, dtype=np.float64)) - 1.0) <= 1e-6
    f, db = response_db(taps, M, n_fft=1 << 21)
    passband = db[np.abs(f) <= 60e3]
    assert passband.min() >= -0.01 and passband.max() <= 0.01
    assert db[np.abs(f) >= 132e3].max() <= -90.0


@pytest.mark.parametrize("M", CHANNELS)
def test_tune_and_place_real_map_back_to_the_frequency(M):
    fs = int(synth.wideband_rate(M))
    rng = np.random.default_rng(11 + M)
    freqs = np.concatenate([rng.integers(0, fs // 2 + 1, 400), [0, 47999, 48000, fs // 2 - 48000, fs // 2]])
    for mode in MIRRORED + PLAIN:
        for f in freqs:
            ch, nco = rx.chan_tune_real(M, mode, float(f))
            f_rel = (nco - 48000) if mode in MIRRORED else -(nco - 48000)
            assert 0 <= ch <= M // 2 and abs(f_rel) <= 48000
            assert ch * 96000 + f_rel == int(f), (mode, f, ch, nco)
            assert rx.chan_centre_real(ch) + f_rel == int(f)
            pch, shift, pnco = rx.chan_place_real(M, mode, float(f))
            assert (pch, pnco) == (ch, 0)
            f_rel = shift - 48000 if mode in MIRRORED else shift + 48000
            assert abs(f_rel) <= 48000 and ch * 96000 + f_rel == int(f), (mode, f, ch, shift)


@pytest.mark.parametrize("M", CHANNELS)
def test_tune_and_place_real_reject_bad_input(M):
    half = synth.wideband_rate(M) / 2
    for fn in (rx.chan_tune_real, rx.chan_place_real):
        for f in (-1.0, -1e-3, half + 1e-3, half + 1, 1e12, float("nan")):
            with pytest.raises(rx.T41RxError, match="_real"):
                fn(M, rx.DEMOD_USB, f)
        for mode in (4, 6, 7, -1, 99):
            with pytest.raises(rx.T41RxError, match="invalid mode"):
                fn(M, mode, 1e6)
        for bad_m in (64, 512, 100, 256, 2048):
            with pytest.raises(rx.T41RxError):
                fn(bad_m, rx.DEMOD_USB, 0.0)


def test_create_checks_the_channel_count_of_each_kind():
    h = C.c_void_p()
    for m in (128, 1024):
        assert rx.lib().t41rx_chan_create(C.byref(h), m, 4, 0) == EINVAL
    for m in (64, 512, 256, 2048):
        assert rx.lib().t41rx_chan_create_real(C.byref(h), m, 4, 0) == EINVAL
    assert not h.value


def test_create_real_without_device_is_enodev():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    h = C.c_void_p()
    assert rx.lib().t41rx_chan_create_real(C.byref(h), 1024, 4, 0) == ENODEV
    assert b"no CUDA device" in rx.lib().t41rx_last_error()
    assert not h.value


# ---------------------------------------------------------------- GPU tier

def _x(capture):
    return capture.astype(np.float64) / 32768.0


def _test_capture(M, n_blocks, seed):
    r = np.random.default_rng(seed)
    fs = synth.wideband_rate(M)
    sig = [("tone", float(r.uniform(0, fs / 2)), {"amp": float(r.uniform(0.03, 0.15))}) for _ in range(6)]
    sig.append(("tone", rx.chan_centre_real(1) + 1234.5, {"amp": 0.1}))
    sig.append(("tone", rx.chan_centre_real(M // 2) - 20000.0, {"amp": 0.1}))
    return synth.wideband_real(seed, M, n_blocks, sig, sigma=0.05)


@pytest.mark.gpu
@pytest.mark.parametrize("M", CHANNELS)
def test_formula_parity_real(M):
    """Channels 0, 1, M/4, M/2 - 1, M/2 and a mapped one, unshifted and with positive, negative and +-96000 Hz shifts,
    an unmapped receiver, over two calls: against float64 z_k[m] exp(2 pi j shift m / 192000) on x = s / 32768, error
    RMS <= 1e-6 of the capture's RMS."""
    n_blocks = 4 if M == 128 else 2
    capture = _test_capture(M, n_blocks, 300 + M)
    chmap = [0, 1, M // 4, M // 2 - 1, M // 2, 7, 7, 1, M // 2, 0, -1]
    shifts = [0, 0, 0, 0, 0, 0, 12345, -54321, 96000, -96000, 777]
    got = channelize(M, len(chmap), capture, [1, n_blocks - 1], [chmap, None], [shifts, None], real=True)
    x, taps = _x(capture), rx.chan_taps(M)
    ref = {k: reference_channel(x, taps, M, k, n_blocks * BLOCK) for k in set(chmap) if k >= 0}
    want = {r: rotate(ref[k], 0, s) for r, (k, s) in enumerate(zip(chmap, shifts)) if k >= 0}
    assert np.all(got[chmap.index(-1)] == 12345.0)
    ratio = error_ratio(got, want, x)
    print("M=%d: error RMS / capture RMS = %.3g" % (M, ratio))
    assert ratio <= 1e-6


@pytest.mark.gpu
def test_split_calls_and_map_changes_are_bit_identical_real():
    """1 + 2 + 5 blocks equal one call, with and without shifts; a map change before the third call gives each
    receiver the bits of its new channel."""
    M, T = 128, 8
    capture = _test_capture(M, T, 5)
    map1 = [3, 40, -1, 3, 64, 0]
    map2 = [40, 3, 64, -1, 0, 3]
    shifts = [48000, -20000, 0, 0, 95999, 777]
    for sh in (None, shifts):
        one = channelize(M, 6, capture, [T], [map1], [sh], real=True)
        split = channelize(M, 6, capture, [1, 2, 5], [map1, None, None], [sh, None, None], real=True)
        assert np.array_equal(one.view(np.uint32), split.view(np.uint32))
        assert np.all(one[2] == 12345.0)
    one = channelize(M, 6, capture, [T], [map1], real=True)
    changed = channelize(M, 6, capture, [1, 2, 5], [map1, None, map2], real=True)
    assert np.array_equal(changed[:, :3].view(np.uint32), one[:, :3].view(np.uint32))
    by_channel = {k: one[r] for r, k in enumerate(map1) if k >= 0}
    for r, k in enumerate(map2):
        if k < 0:
            assert np.all(changed[r, 3:] == 12345.0)
        else:
            assert np.array_equal(changed[r, 3:].view(np.uint32), by_channel[k][3:].view(np.uint32)), r


@pytest.mark.gpu
@pytest.mark.parametrize("M, k", [(128, 5), (128, 57), (1024, 146)])
def test_real_tone_gain_and_rejection(M, k):
    """A cos(2 pi f t) at the centre of channel k: |z| = A / 2 +- 0.01 dB there, <= -90 dB two channels away and
    further (after the first block, the filter's start-up)."""
    T, amp = 3, 0.5
    capture = synth.wideband_real(0, M, T, [("tone", rx.chan_centre_real(k), {"amp": amp})])
    got = channelize(M, M // 2 + 1, capture, [T], [list(range(M // 2 + 1))], real=True)[:, 1:]
    level = 20.0 * np.log10(np.sqrt(np.mean(got.astype(np.float64) ** 2 * 2, axis=(1, 2, 3))) / (amp / 2))
    print("M=%d k=%d: %.4f dB at the channel, worst %.1f dB two or more away" %
          (M, k, level[k], max(level[j] for j in range(M // 2 + 1) if abs(j - k) >= 2)))
    assert abs(level[k]) <= 0.01, level[k]
    far = [j for j in range(M // 2 + 1) if abs(j - k) >= 2]
    assert level[far].max() <= -90.0, level[far].max()


@pytest.mark.gpu
def test_argument_checks_real():
    import torch
    M = 128
    cap = torch.zeros(BLOCK * M // 2 + 16, dtype=torch.int16, device="cuda")
    iq = torch.zeros((2, 1, BLOCK, 2), dtype=torch.float32, device="cuda")
    cap_f = torch.zeros((BLOCK * 32, 2), dtype=torch.float32, device="cuda")
    with rx.Channelizer(M, 2, real=True) as ch:
        ch.set_map([M // 2, 0])
        with pytest.raises(rx.T41RxError, match="channel out of range"):
            ch.set_map([M // 2 + 1, 0])
        for off in (2, 8):           # 2-byte and 8-byte aligned, not 16
            with pytest.raises(rx.T41RxError, match="aligned"):
                ch.process_device(cap.data_ptr() + off, iq.data_ptr(), 1)
        assert rx.lib().t41rx_chan_process_device(ch._h, cap_f.data_ptr(), iq.data_ptr(), 1, None) == EINVAL
        ch.process_device(cap.data_ptr(), iq.data_ptr(), 1)
        ch.synchronize()
    with rx.Channelizer(64, 2) as ch:
        ch.set_map([0, 1])
        assert rx.lib().t41rx_chan_process_device_real(ch._h, cap.data_ptr(), iq.data_ptr(), 1, None) == EINVAL
    h = C.c_void_p()
    assert rx.lib().t41rx_chan_create(C.byref(h), 128, 4, 0) == EINVAL


@pytest.mark.gpu
def test_sideband_at_a_channel_centre_real():
    """A tone 1 kHz above a USB dial at the centre of channel 147 (14.112 MHz) of M = 1024, placed by
    chan_place_real: 1 kHz audio in USB and >= 65 dB weaker in LSB."""
    M, T = 1024, 8
    dial = rx.chan_centre_real(147)
    placed = rx.chan_place_real(M, rx.DEMOD_USB, dial)
    assert placed == rx.chan_place_real(M, rx.DEMOD_LSB, dial) == (147, 48000, 0)
    ch, shift, nco = placed
    capture = synth.wideband_real(1, M, T, [("tone", dial + 1000.0, {"amp": 0.2})])
    iq = channelize(M, 2, capture, [T], [[ch, ch]], [[shift, shift]], real=True)
    ps = [rx.make_params(mode=rx.DEMOD_USB, nco_freq=nco, agc_mode=0),
          rx.make_params(mode=rx.DEMOD_LSB, nco_freq=nco, agc_mode=0)]
    audio = chain(ps, iq)["audio"][:, 4:].reshape(2, -1).astype(np.float64)
    spec = np.abs(np.fft.rfft(audio[0] * np.hanning(audio.shape[1])))
    f_peak = np.argmax(spec) * 192000.0 / audio.shape[1]
    assert abs(f_peak - 1000.0) <= 2 * 192000.0 / audio.shape[1], f_peak
    ratio = 10 * np.log10(np.mean(audio[0] ** 2) / max(np.mean(audio[1] ** 2), 1e-300))
    print("USB / LSB %.1f dB" % ratio)
    assert ratio >= 65.0


def _psk_through_the_channelizer(M, freq, step):
    """PSK31 at freq (Hz from 0) placed by chan_place_real; the capture is generated and channelized `step` blocks at
    a time (a long capture at up to 98 MS/s); returns the decoded characters"""
    import torch
    ch, shift, nco = rx.chan_place_real(M, rx.DEMOD_USB, freq)
    T = synth.psk31_blocks(cases.PSK_TEXT, 5014)
    signals = [("psk31", freq, {"amp": 0.25, "text": cases.PSK_TEXT, "symbol_offset": 5014})]
    iq = torch.empty((1, T, BLOCK, 2), dtype=torch.float32, device="cuda")
    with rx.Channelizer(M, 1, real=True) as chan:
        chan.set_map([ch])
        chan.set_shift([shift])
        for b0 in range(0, T, step):
            nb = min(step, T - b0)
            cap = torch.from_numpy(synth.wideband_real(31, M, nb, signals, sigma=0.01, start_block=b0)).cuda()
            # one receiver: the call's [1][nb][2048][2] output is the buffer from block b0 on
            chan.process_device(cap.data_ptr(), iq[0, b0].data_ptr(), nb)
            chan.synchronize()
    ps =[rx.make_params(mode=rx.DEMOD_USB, f_lo_cut=-100, f_hi_cut=100, agc_mode=0, psk31_enable=1, nco_freq=nco)]
    out = chain(ps, iq.cpu().numpy(), want_psk=True)
    return bytes(out["psk_chars"][0][out["psk_chars"][0] > 0])


@pytest.mark.gpu
@pytest.mark.parametrize("M, freq", [(1024, 14.140e6), (128, 3.580e6)])
def test_psk31_decodes_real(M, freq):
    """PSK31 on 20 m (14.140 MHz, M = 1024) and on 80 m (3.580 MHz, M = 128), placed by chan_place_real, both 28 kHz
    above their channel's centre.  (At 14.070 MHz, 42 kHz below the centre of channel 147, the placement rule of
    chan_place does not decode PSK31, through the complex path on the oracle as well: DESIGN section 3.8.)"""
    chars = _psk_through_the_channelizer(M, freq, 16 if M == 1024 else 67)
    assert cases.PSK_TEXT.encode() in chars, chars


@pytest.mark.gpu
def test_bank_placed_by_chan_place_real_matches_rotated_reference_feed():
    """32 receivers (USB, LSB, AM, NFM, PSK31-in-USB) across 0 - 6.144 MHz of an M = 128 capture, placed by
    chan_place_real: the chain on the channelizer's output and on the rotated float64 reference (x = s / 32768) rounded
    to float32 (flags = 0 both): audio SNR >= 90 dB after block 2, discrete state identical."""
    M, T, n = 128, 12, 32
    r = np.random.default_rng(33)
    half = synth.wideband_rate(M) / 2
    signals, params, chmap, shifts = [], [], [], []
    for i in range(n):
        f = (i + 0.5) * half / n + float(r.uniform(-20e3, 20e3))
        kind = i % 5
        amp = 0.02                       # 32 signals stay inside int16 full scale
        if kind == 0:
            mode, sig = rx.DEMOD_USB, ("tone", f + float(r.uniform(400, 2600)), {"amp": amp})
        elif kind == 1:
            mode, sig = rx.DEMOD_LSB, ("tone", f - float(r.uniform(400, 2600)), {"amp": amp})
        elif kind == 2:
            mode, sig = rx.DEMOD_AM, ("am", f, {"amp": amp})
        elif kind == 3:
            mode, sig = rx.DEMOD_NFM, ("nfm", f, {"amp": amp})
        else:
            mode, sig = rx.DEMOD_USB, ("psk31", f, {"amp": amp, "text": cases.PSK_TEXT, "symbol_offset": 5014})
        ch, shift, nco = rx.chan_place_real(M, mode, f)
        signals.append(sig)
        chmap.append(ch)
        shifts.append(shift)
        if kind == 4:
            params.append(rx.make_params(mode=mode, f_lo_cut=-100, f_hi_cut=100, agc_mode=0, psk31_enable=1, nco_freq=nco))
        elif kind == 3:
            params.append(rx.make_params(mode=mode, nco_freq=nco, nfm_filter_bw=12000))
        else:
            params.append(rx.make_params(mode=mode, nco_freq=nco))
    capture = synth.wideband_real(9, M, T, signals, sigma=0.002)
    assert np.abs(capture).max() < 32767
    got_iq = channelize(M, n, capture, [T], [chmap], [shifts], real=True)
    x, taps = _x(capture), rx.chan_taps(M)
    ref_iq = np.empty_like(got_iq)
    for s, (k, sh) in enumerate(zip(chmap, shifts)):
        z = rotate(reference_channel(x, taps, M, k, T * BLOCK), 0, sh)
        ref_iq[s, ..., 0] = z.real.reshape(T, BLOCK)
        ref_iq[s, ..., 1] = z.imag.reshape(T, BLOCK)
    got, want = chain(params, got_iq), chain(params, ref_iq)
    worst = np.inf
    for s in range(n):
        snr = O.snr_db(want["audio"][s, 2:], got["audio"][s, 2:])
        worst = min(worst, snr)
        assert snr >= 90.0, (s, snr)
        for f in cases.DEBUG_INT_FIELDS:
            assert getattr(got["debug"][s], f) == getattr(want["debug"][s], f), (s, f)
    print("worst audio SNR %.1f dB" % worst)
