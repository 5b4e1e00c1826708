"""Polyphase channelizer (t41rx_chan_*): one wideband capture at M x 96 kS/s cut into the receivers' 192 kS/s blocks.

CPU tier: the prototype's design (symmetry, DC gain, passband ripple, stopband), where t41rx_chan_tune puts a
receiver, and the refusal without a GPU.  GPU tier: the kernel against a float64 evaluation of the defining formula,
bit-identity across call splits and map changes, the stopband seen through the kernel, the sideband convention end to
end through the chain, a receiver bank fed by the channelizer against the same bank fed by the reference, and PSK31
decoded through the wideband path.
"""
import numpy as np
import pytest

import cases
import oracle_py as O
from chan_driver import chain, channelize, cplx, reference_channel, response_db
from t41_sdr_b200 import rx, synth

CHANNELS = (64, 512)
MIRRORED = (rx.DEMOD_USB, rx.DEMOD_LSB, rx.DEMOD_AM, rx.DEMOD_SAM)
PLAIN = (rx.DEMOD_NFM, rx.DEMOD_PSK31)
BLOCK = rx.BLOCK


# ---------------------------------------------------------------- CPU tier

@pytest.mark.parametrize("M", CHANNELS)
def test_prototype_design(M):
    taps = rx.chan_taps(M)
    assert taps.dtype == np.float32 and taps.size == 10 * M
    assert np.array_equal(taps, taps[::-1])
    assert abs(float(np.sum(taps, dtype=np.float64)) - 1.0) <= 1e-6
    f, db = response_db(taps, M)
    passband = db[np.abs(f) <= 60e3]
    assert passband.min() >= -0.01 and passband.max() <= 0.01
    assert db[np.abs(f) >= 132e3].max() <= -90.0


@pytest.mark.parametrize("M", CHANNELS)
def test_tune_maps_back_to_the_offset(M):
    fs = int(synth.wideband_rate(M))
    rng = np.random.default_rng(7 + M)
    offsets = np.concatenate([rng.integers(-fs // 2, fs // 2, 400),
                              [-fs // 2, fs // 2 - 1, 0, 48000, -48000, 47999, 96000, 144000, fs // 2 - 48000,
                               fs // 2 - 48001, -fs // 2 + 48000]])
    for mode in MIRRORED + PLAIN:
        for off in offsets:
            ch, nco = rx.chan_tune(M, mode, float(off))
            assert 0 <= ch < M
            f_rel = (nco - 48000) if mode in MIRRORED else -(nco - 48000)
            assert abs(f_rel) <= 48000
            # the capture's spectrum is periodic in Fs_in: channel M/2 (centre -Fs_in/2) also holds +Fs_in/2
            assert (rx.chan_centre(M, ch) + f_rel - int(off)) % fs == 0, (mode, off, ch, nco)


@pytest.mark.parametrize("M", CHANNELS)
def test_tune_rejects_out_of_band_and_bad_modes(M):
    half = synth.wideband_rate(M) / 2
    for off in (half, half + 1, -half - 1, 1e12, float("nan")):
        with pytest.raises(rx.T41RxError):
            rx.chan_tune(M, rx.DEMOD_USB, off)
    for mode in (4, 6, 7, -1, 99):
        with pytest.raises(rx.T41RxError):
            rx.chan_tune(M, mode, 0.0)
    with pytest.raises(rx.T41RxError):
        rx.chan_tune(128, rx.DEMOD_USB, 0.0)
    with pytest.raises(rx.T41RxError):
        rx.chan_taps(100)


def test_create_without_device_is_enodev():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    import ctypes as C
    h = C.c_void_p()
    assert rx.lib().t41rx_chan_create(C.byref(h), 64, 4, 0) == -4    # T41RX_ENODEV
    assert b"no CUDA device" in rx.lib().t41rx_last_error()
    assert not h.value


# ---------------------------------------------------------------- GPU tier

def _test_capture(M, n_blocks, seed):
    r = np.random.default_rng(seed)
    fs = synth.wideband_rate(M)
    sig = [("tone", float(r.uniform(-fs / 2, fs / 2)), {"amp": float(r.uniform(0.05, 0.5))}) for _ in range(6)]
    sig.append(("tone", rx.chan_centre(M, 1) + 1234.5, {"amp": 0.3}))
    return synth.wideband(seed, M, n_blocks, sig, sigma=0.2)


@pytest.mark.gpu
@pytest.mark.parametrize("M", CHANNELS)
def test_formula_parity(M):
    """Measured on a B200: error RMS 1.58e-8 (M = 64) and 1.11e-8 (M = 512) of the capture's RMS (limit 1e-6)."""
    n_blocks = 4 if M == 64 else 2
    capture = _test_capture(M, n_blocks, 100 + M)
    check = sorted({0, 1, M // 2 - 1, M // 2, M - 1, 7, M // 2 + 5})
    chmap = check + [7, -1]
    got = channelize(M, len(chmap), capture, [1, n_blocks - 1], [chmap, None])
    taps = rx.chan_taps(M)
    x = cplx(capture)
    n_out = n_blocks * BLOCK
    err2 = 0.0
    for r, k in enumerate(chmap):
        if k < 0:
            assert np.all(got[r] == 12345.0)
            continue
        want = reference_channel(x, taps, M, k, n_out)
        g = got[r].reshape(n_out, 2)
        err2 += np.sum((g[:, 0] - want.real) ** 2 + (g[:, 1] - want.imag) ** 2)
    n_vals = sum(1 for k in chmap if k >= 0) * n_out
    ratio = np.sqrt(err2 / n_vals) / np.sqrt(np.mean(np.abs(x) ** 2))
    print("M=%d: error RMS / capture RMS = %.3g" % (M, ratio))
    assert ratio <= 1e-6


@pytest.mark.gpu
def test_split_calls_and_map_changes_are_bit_identical():
    M, T = 64, 8
    capture = _test_capture(M, T, 5)
    map1 = [3, 40, -1, 3, 63, 32]
    map2 = [40, 3, 63, -1, 32, 3]
    one = channelize(M, 6, capture, [T], [map1])
    split = channelize(M, 6, capture, [1, 2, 5], [map1, None, None])
    assert np.array_equal(one.view(np.uint32), split.view(np.uint32))
    assert np.all(one[2] == 12345.0)                                   # unmapped: sentinel kept
    assert np.array_equal(one[0].view(np.uint32), one[3].view(np.uint32))   # a shared channel: identical copies
    changed = channelize(M, 6, capture, [1, 2, 5], [map1, None, map2])
    assert np.array_equal(changed[:, :3].view(np.uint32), one[:, :3].view(np.uint32))
    by_channel = {k: one[r] for r, k in enumerate(map1) if k >= 0}
    for r, k in enumerate(map2):
        if k < 0:
            assert np.all(changed[r, 3:] == 12345.0)
        else:
            assert np.array_equal(changed[r, 3:].view(np.uint32), by_channel[k][3:].view(np.uint32)), r


@pytest.mark.gpu
@pytest.mark.parametrize("k", [5, 33])
def test_stopband_through_the_kernel(k):
    M, T, amp = 64, 3, 0.5
    capture = synth.wideband(0, M, T, [("tone", rx.chan_centre(M, k), {"amp": amp})])
    got = channelize(M, M, capture, [T], [list(range(M))])[:, 1:]     # after the first block (the filter's start-up)
    level = 20.0 * np.log10(np.sqrt(np.mean(got.astype(np.float64) ** 2 * 2, axis=(1, 2, 3))) / amp)
    assert abs(level[k]) <= 0.01, level[k]
    far = [j for j in range(M) if min((j - k) % M, (k - j) % M) >= 2]
    assert level[far].max() <= -90.0, level[far].max()


@pytest.mark.gpu
def test_sideband_convention_end_to_end():
    """A tone 1 kHz above a USB dial point placed by chan_tune is 1 kHz audio in USB and >= 60 dB weaker in LSB.
    The dial sits 43.6 kHz below its channel centre (NCOFreq 4433): the chain's own opposite-sideband rejection depends
    on NCOFreq (fed directly at 192 kS/s: 72 dB at 0, 19 dB at 48000; DESIGN section 3.7).  Measured on a B200 through
    the channelizer at NCOFreq 61433: 51.3 dB, the chain fed directly there: 52.6 dB."""
    M, T, dial = 64, 8, -1291567.0
    ch_u, nco_u = rx.chan_tune(M, rx.DEMOD_USB, dial)
    ch_l, nco_l = rx.chan_tune(M, rx.DEMOD_LSB, dial)
    assert (ch_u, nco_u) == (ch_l, nco_l) == (M - 13, 4433)
    capture = synth.wideband(1, M, T, [("tone", dial + 1000.0, {"amp": 0.1})])
    iq = channelize(M, 2, capture, [T], [[ch_u, ch_l]])
    ps = [rx.make_params(mode=rx.DEMOD_USB, nco_freq=nco_u, agc_mode=0),
          rx.make_params(mode=rx.DEMOD_LSB, nco_freq=nco_l, agc_mode=0)]
    audio = chain(ps, iq)["audio"][:, 4:].reshape(2, -1).astype(np.float64)
    spec = np.abs(np.fft.rfft(audio[0] * np.hanning(audio.shape[1])))
    f_peak = np.argmax(spec) * 192000.0 / audio.shape[1]
    assert abs(f_peak - 1000.0) <= 2 * 192000.0 / audio.shape[1], f_peak
    p_usb, p_lsb = np.mean(audio[0] ** 2), np.mean(audio[1] ** 2)
    assert p_usb > 0 and 10 * np.log10(p_usb / max(p_lsb, 1e-300)) >= 60.0


@pytest.mark.gpu
def test_bank_fed_by_channelizer_matches_reference_feed():
    """32 receivers (USB, LSB, AM, NFM, PSK31-in-USB) on one M = 64 capture: the chain on the channelizer's output and
    on the float64 reference's output rounded to float32 (flags = 0 both): audio SNR >= 90 dB after block 2, discrete
    state identical."""
    M, T, n = 64, 12, 32
    r = np.random.default_rng(32)
    fs = synth.wideband_rate(M)
    signals, params, chmap = [], [], []
    for i in range(n):
        f = -fs / 2 + (i + 0.5) * fs / n + float(r.uniform(-20e3, 20e3))
        kind = i % 5
        if kind == 0:
            mode, sig = rx.DEMOD_USB, ("tone", f + float(r.uniform(400, 2600)), {"amp": 0.1})
        elif kind == 1:
            mode, sig = rx.DEMOD_LSB, ("tone", f - float(r.uniform(400, 2600)), {"amp": 0.1})
        elif kind == 2:
            mode, sig = rx.DEMOD_AM, ("am", f, {"amp": 0.1})
        elif kind == 3:
            mode, sig = rx.DEMOD_NFM, ("nfm", f, {"amp": 0.1})
        else:
            mode, sig = rx.DEMOD_USB, ("psk31", f, {"amp": 0.1, "text": cases.PSK_TEXT, "symbol_offset": 5014})
        ch, nco = rx.chan_tune(M, mode, f)
        signals.append(sig)
        chmap.append(ch)
        if kind == 4:
            params.append(rx.make_params(mode=mode, f_lo_cut=-100, f_hi_cut=100, agc_mode=0, psk31_enable=1, nco_freq=nco))
        elif kind == 3:
            params.append(rx.make_params(mode=mode, nco_freq=nco, nfm_filter_bw=12000))
        else:
            params.append(rx.make_params(mode=mode, nco_freq=nco))
    capture = synth.wideband(9, M, T, signals, sigma=0.002)
    got_iq = channelize(M, n, capture, [T], [chmap])
    x, taps = cplx(capture), rx.chan_taps(M)
    ref_iq = np.empty_like(got_iq)
    for s, k in enumerate(chmap):
        z = reference_channel(x, taps, M, k, T * BLOCK)
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


@pytest.mark.gpu
def test_psk31_decodes_through_the_wideband_path():
    """Two PSK31 receivers, on channel 7 and on channel M - 16 (a negative offset), 40 kHz from their centres: the
    chain decodes PSK31 only toward the ends of the NCOFreq range (fed directly at 192 kS/s: at 0, 12000, 84000, 96000,
    not at 24000 ... 72000; DESIGN section 3.7)."""
    M = 64
    offsets = (632123.0, -1495679.0)
    chs = [rx.chan_tune(M, rx.DEMOD_USB, f) for f in offsets]
    assert chs == [(7, 8123), (M - 16, 88321)]
    T = synth.psk31_blocks(cases.PSK_TEXT, 5014)
    signals = [("psk31", f, {"amp": 0.25, "text": cases.PSK_TEXT, "symbol_offset": 5014}) for f in offsets]
    pieces, step = [], 67
    for b0 in range(0, T, step):           # generated and channelized piece by piece: the capture is long
        nb = min(step, T - b0)
        pieces.append(synth.wideband(31, M, nb, signals, sigma=0.01, start_block=b0))
    capture = np.concatenate(pieces)
    calls = [min(step, T - b0) for b0 in range(0, T, step)]
    iq = channelize(M, 2, capture, calls, [[c for c, _ in chs]] + [None] * (len(calls) - 1))
    ps = [rx.make_params(mode=rx.DEMOD_USB, f_lo_cut=-100, f_hi_cut=100, agc_mode=0, psk31_enable=1, nco_freq=nco)
          for _, nco in chs]
    out = chain(ps, iq, want_psk=True)
    for s in range(2):
        chars = bytes(out["psk_chars"][s][out["psk_chars"][s] > 0])
        assert cases.PSK_TEXT.encode() in chars, (s, chars)
