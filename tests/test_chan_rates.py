"""Channelizer at digitizers' native clocks (DESIGN §3.10): complex captures (float and int16 pairs) at M = 320 and 640
(30.72 and 61.44 MS/s, the LTE-family rates), real int16 captures at M = 800 and 1280 (76.8 MS/s, Hermes-Lite 2; 122.88
MS/s, the HPSDR family's ADC clock).  Their row FFTs (320, 400, 640 points) run mixed-radix passes (radix 5 beside 8).

CPU tier: the prototype at each new M, where chan_tune / chan_place (320, 640) and chan_tune_real / chan_place_real (800,
1280) put a receiver, the refusals at creation and in placement, ENODEV without a device.  GPU tier, at every new
(kind, M): the kernel against the float64 defining formula with and without shifts, bit-identity across call splits and
map changes (and for q15, with the float channelizer on s / 32768), a tone's gain and rejection, argument checks; the
chain end to end on receivers placed in M = 640, 800 and 1280 captures.
"""
import ctypes as C

import numpy as np
import pytest

import cases
import oracle_py as O
from chan_driver import chain, channelize, cplx, error_ratio, reference_channel, response_db, rotate
from t41_sdr_b200 import rx, synth

COMPLEX = (320, 640)
REAL = (800, 1280)
MIRRORED = (rx.DEMOD_USB, rx.DEMOD_LSB, rx.DEMOD_AM, rx.DEMOD_SAM)
PLAIN = (rx.DEMOD_NFM, rx.DEMOD_PSK31)
KINDS = [("float", m) for m in COMPLEX] + [("q15", m) for m in COMPLEX] + [("real", m) for m in REAL]
BLOCK = rx.BLOCK
EINVAL, ENODEV = -1, -4
FILL = 12345.0


# ---------------------------------------------------------------- CPU tier

@pytest.mark.parametrize("M", COMPLEX + REAL)
def test_prototype_design_at_new_rates(M):
    taps = rx.chan_taps(M)
    assert taps.dtype == np.float32 and taps.size == 10 * M
    assert np.array_equal(taps, taps[::-1])
    assert abs(float(np.sum(taps, dtype=np.float64)) - 1.0) <= 1e-6
    f, db = response_db(taps, M, n_fft=1 << 21)
    passband = db[np.abs(f) <= 60e3]
    assert passband.min() >= -0.01 and passband.max() <= 0.01
    assert db[np.abs(f) >= 132e3].max() <= -90.0


@pytest.mark.parametrize("M", COMPLEX)
def test_tune_and_place_map_back_to_the_offset(M):
    fs = int(synth.wideband_rate(M))
    rng = np.random.default_rng(17 + M)
    offsets = np.concatenate([rng.integers(-fs // 2, fs // 2, 400),
                              [-fs // 2, fs // 2 - 1, 0, 48000, -48000, 47999, 96000, 144000, fs // 2 - 48000,
                               fs // 2 - 48001, -fs // 2 + 48000]])
    for mode in MIRRORED + PLAIN:
        for off in offsets:
            ch, nco = rx.chan_tune(M, mode, float(off))
            assert 0 <= ch < M
            f_rel = (nco - 48000) if mode in MIRRORED else -(nco - 48000)
            assert abs(f_rel) <= 48000
            assert (rx.chan_centre(M, ch) + f_rel - int(off)) % fs == 0, (mode, off, ch, nco)
            pch, shift, pnco = rx.chan_place(M, mode, float(off))
            assert (pch, pnco) == (ch, 0)
            f_rel = shift - 48000 if mode in MIRRORED else shift + 48000
            assert abs(f_rel) <= 48000
            assert (rx.chan_centre(M, ch) + f_rel - int(off)) % fs == 0, (mode, off, ch, shift)


@pytest.mark.parametrize("M", REAL)
def test_tune_and_place_real_map_back_to_the_frequency_at_new_rates(M):
    fs = int(synth.wideband_rate(M))
    rng = np.random.default_rng(19 + M)
    freqs = np.concatenate([rng.integers(0, fs // 2 + 1, 400), [0, 47999, 48000, fs // 2 - 48000, fs // 2]])
    for mode in MIRRORED + PLAIN:
        for f in freqs:
            ch, nco = rx.chan_tune_real(M, mode, float(f))
            f_rel = (nco - 48000) if mode in MIRRORED else -(nco - 48000)
            assert 0 <= ch <= M // 2 and abs(f_rel) <= 48000
            assert ch * 96000 + f_rel == int(f), (mode, f, ch, nco)
            pch, shift, pnco = rx.chan_place_real(M, mode, float(f))
            assert (pch, pnco) == (ch, 0)
            f_rel = shift - 48000 if mode in MIRRORED else shift + 48000
            assert abs(f_rel) <= 48000 and ch * 96000 + f_rel == int(f), (mode, f, ch, shift)


def test_placement_rejects_the_other_kinds_channel_counts():
    for m in REAL + (128, 1024):
        for fn in (rx.chan_tune, rx.chan_place):
            with pytest.raises(rx.T41RxError):
                fn(m, rx.DEMOD_USB, 0.0)
    for m in COMPLEX + (64, 512):
        for fn in (rx.chan_tune_real, rx.chan_place_real):
            with pytest.raises(rx.T41RxError):
                fn(m, rx.DEMOD_USB, 0.0)
    for m in (100, 400, 480, 960, 1600):
        with pytest.raises(rx.T41RxError, match="320, 512, 640, 800"):
            rx.chan_taps(m)


def test_create_checks_the_channel_count_of_each_kind_at_new_rates():
    h = C.c_void_p()
    for create in ("t41rx_chan_create", "t41rx_chan_create_q15"):
        for m in (800, 1280, 400, 480, 960, 100):
            assert getattr(rx.lib(), create)(C.byref(h), m, 4, 0) == EINVAL
            assert b"64, 320, 512 or 640" in rx.lib().t41rx_last_error()
    for m in (320, 640, 400, 960, 1600):
        assert rx.lib().t41rx_chan_create_real(C.byref(h), m, 4, 0) == EINVAL
        assert b"128, 800, 1024 or 1280" in rx.lib().t41rx_last_error()
    assert not h.value


@pytest.mark.parametrize("kind, M", KINDS)
def test_create_at_new_rates_without_device_is_enodev(kind, M):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    create = {"float": "t41rx_chan_create", "q15": "t41rx_chan_create_q15", "real": "t41rx_chan_create_real"}[kind]
    h = C.c_void_p()
    assert getattr(rx.lib(), create)(C.byref(h), M, 4, 0) == ENODEV
    assert b"no CUDA device" in rx.lib().t41rx_last_error()
    assert not h.value


# ---------------------------------------------------------------- GPU tier

def _capture(kind, M, n_blocks, seed):
    """a seeded capture of the kind: six random tones, one near the top channel's centre, noise; for q15 full-scale
    samples (-32768 and 32767, in I and in Q) scattered through it"""
    r = np.random.default_rng(seed)
    fs = synth.wideband_rate(M)
    if kind == "real":
        sig = [("tone", float(r.uniform(0, fs / 2)), {"amp": float(r.uniform(0.03, 0.15))}) for _ in range(6)]
        sig.append(("tone", rx.chan_centre_real(M // 2) - 20000.0, {"amp": 0.1}))
        return synth.wideband_real(seed, M, n_blocks, sig, sigma=0.05)
    sig = [("tone", float(r.uniform(-fs / 2, fs / 2)), {"amp": float(r.uniform(0.03, 0.15))}) for _ in range(6)]
    sig.append(("tone", rx.chan_centre(M, M // 2) + 1234.5, {"amp": 0.1}))
    if kind == "float":
        return synth.wideband(seed, M, n_blocks, sig, sigma=0.05)
    s = synth.wideband_q15(seed, M, n_blocks, sig, sigma=0.05)
    for value in (-32768, 32767):
        idx = r.choice(s.shape[0], 64, replace=False)
        s[idx, r.integers(0, 2, idx.size)] = value
        s[r.choice(s.shape[0], 8, replace=False)] = value
    return s


def _x(kind, capture):
    """the capture as the channelizer reads it, complex128"""
    if kind == "real":
        return capture.astype(np.float64) / 32768.0
    return cplx(capture) / (32768.0 if kind == "q15" else 1.0)


def _opts(kind):
    return {"real": kind == "real", "q15": kind == "q15"}


def _last(kind, M):
    return M // 2 if kind == "real" else M - 1


@pytest.mark.gpu
@pytest.mark.parametrize("kind, M", KINDS)
def test_formula_parity_at_new_rates(kind, M):
    """Channels 0, 1, M/5 (a multiple of the radix-5 stride), M/2 - 1, M/2, the last one (M - 1, or M/2 for real) and a
    mapped one (7), unshifted and with positive, negative, +-96000 and +-191999 Hz shifts (two on channel 7), an
    unmapped receiver, over two calls: against float64 z_k[m] exp(2 pi j shift m / 192000), error RMS <= 1e-6 of the
    capture's RMS."""
    n_blocks = 2
    capture = _capture(kind, M, n_blocks, 500 + M)
    chmap = [0, 1, M // 5, M // 2 - 1, M // 2, _last(kind, M), 7, 7, 1, M // 2, 0, M // 5, -1]
    shifts = [0, 0, 0, 0, 0, 0, 12345, -54321, 96000, -96000, 191999, -191999, 777]
    got = channelize(M, len(chmap), capture, [1, n_blocks - 1], [chmap, None], [shifts, None], **_opts(kind))
    x, taps = _x(kind, capture), rx.chan_taps(M)
    ref = {k: reference_channel(x, taps, M, k, n_blocks * BLOCK) for k in set(chmap) if k >= 0}
    want = {r: rotate(ref[k], 0, s) for r, (k, s) in enumerate(zip(chmap, shifts)) if k >= 0}
    assert np.all(got[chmap.index(-1)] == FILL)
    ratio = error_ratio(got, want, x)
    print("%s M=%d: error RMS / capture RMS = %.3g" % (kind, M, ratio))
    assert ratio <= 1e-6


@pytest.mark.gpu
@pytest.mark.parametrize("kind, M", KINDS)
def test_split_calls_and_map_changes_are_bit_identical_at_new_rates(kind, M):
    """1 + 2 + 5 blocks equal one 8-block call, with and without shifts; a map change before the third call (receivers
    unmapped, an unmapped one mapped) gives each receiver the bits of its new channel."""
    T, last = 8, _last(kind, M)
    capture = _capture(kind, M, T, 50 + M)
    map1 = [0, 1, M // 5, last, 5, 5, -1, 3]
    map2 = [5, -1, 0, last, M // 5, 3, 1, -1]
    shifts = [48000, -20000, 0, 0, 95999, -191999, 777, 191999]
    for sh in (None, shifts):
        one = channelize(M, 8, capture, [T], [map1], [sh], **_opts(kind))
        split = channelize(M, 8, capture, [1, 2, 5], [map1, None, None], [sh, None, None], **_opts(kind))
        assert np.array_equal(one.view(np.uint32), split.view(np.uint32))
        assert np.all(one[6] == FILL)
    one = channelize(M, 8, capture, [T], [map1], **_opts(kind))
    assert np.array_equal(one[4].view(np.uint32), one[5].view(np.uint32))     # a shared channel: identical copies
    changed = channelize(M, 8, capture, [1, 2, 5], [map1, None, map2], **_opts(kind))
    assert np.array_equal(changed[:, :3].view(np.uint32), one[:, :3].view(np.uint32))
    by_channel = {k: one[r] for r, k in enumerate(map1) if k >= 0}
    for r, k in enumerate(map2):
        if k < 0:
            assert np.all(changed[r, 3:] == FILL), r
        else:
            assert np.array_equal(changed[r, 3:].view(np.uint32), by_channel[k][3:].view(np.uint32)), r


@pytest.mark.gpu
@pytest.mark.parametrize("M", COMPLEX)
def test_q15_is_bit_identical_to_float_at_new_rates(M):
    """A q15 channelizer on s and a float channelizer on s / 32768 (exact) run the same schedule: calls of 1 + 2 + 5
    blocks, a map change before the third call (receivers unmapped and remapped), shifts set before the first and the
    second call (positive, negative, +-96000, +-191999, two shifts on one channel), receivers 7 ... 9 never shifted."""
    capture = _capture("q15", M, 8, 40 + M)
    assert (capture == -32768).any() and (capture == 32767).any()
    map1 = [0, 1, M // 5, M // 2, M - 1, 5, 5, -1, 3, 7]
    map2 = [5, -1, 0, M - 1, M // 2, 5, 3, 2, -1, M // 5]
    shifts1 = [12345, -54321, 96000, -96000, 0, 777, -191999]
    shifts2 = [191999, -191999, 4000, 0]
    calls, maps, shifts = [1, 2, 5], [map1, None, map2], [shifts1, shifts2, None]
    got = channelize(M, len(map1), capture, calls, maps, shifts, q15=True)
    want = channelize(M, len(map1), capture.astype(np.float32) / 32768.0, calls, maps, shifts)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    assert np.all(got[7, :3] == FILL)
    assert np.all(got[1, 3:] == FILL) and np.all(got[8, 3:] == FILL)
    for r in (0, 2, 3, 4, 5, 6, 9):
        assert not np.any(got[r] == FILL), r


@pytest.mark.gpu
@pytest.mark.parametrize("kind, M, k", [("float", 320, 67), ("float", 640, 131), ("q15", 640, 509),
                                        ("real", 800, 37), ("real", 1280, 147)])
def test_tone_gain_and_rejection_at_new_rates(kind, M, k):
    """A tone at the centre of channel k (complex: exp(2 pi j f t); real: cos(2 pi f t)): |z| = A (real: A / 2)
    +- 0.01 dB there, <= -90 dB two channels away and further (after the first block, the filter's start-up)."""
    T, amp = 3, 0.5
    if kind == "real":
        n_ch, gain = M // 2 + 1, amp / 2
        capture = synth.wideband_real(0, M, T, [("tone", rx.chan_centre_real(k), {"amp": amp})])
        far = [j for j in range(n_ch) if abs(j - k) >= 2]
    else:
        n_ch, gain = M, amp
        sig = [("tone", rx.chan_centre(M, k), {"amp": amp})]
        capture = synth.wideband(0, M, T, sig) if kind == "float" else synth.wideband_q15(0, M, T, sig)
        far = [j for j in range(M) if min((j - k) % M, (k - j) % M) >= 2]
    got = channelize(M, n_ch, capture, [T], [list(range(n_ch))], **_opts(kind))[:, 1:]
    level = 20.0 * np.log10(np.sqrt(np.mean(got.astype(np.float64) ** 2 * 2, axis=(1, 2, 3))) / gain)
    print("%s M=%d k=%d: %.4f dB at the channel, worst %.1f dB two or more away" % (kind, M, k, level[k], level[far].max()))
    assert abs(level[k]) <= 0.01, level[k]
    assert level[far].max() <= -90.0, level[far].max()


@pytest.mark.gpu
@pytest.mark.parametrize("kind, M", KINDS)
def test_argument_checks_at_new_rates(kind, M):
    import torch
    per_block = BLOCK * M // 2
    if kind == "float":
        cap, offs = torch.zeros((per_block + 8, 2), dtype=torch.float32, device="cuda"), (4,)
    elif kind == "q15":
        cap, offs = torch.zeros((per_block + 8, 2), dtype=torch.int16, device="cuda"), (4, 8)
    else:
        cap, offs = torch.zeros(per_block + 16, dtype=torch.int16, device="cuda"), (2, 8)
    iq = torch.zeros((2, 1, BLOCK, 2), dtype=torch.float32, device="cuda")
    last = _last(kind, M)
    with rx.Channelizer(M, 2, **_opts(kind)) as ch:
        ch.set_map([last, 0])
        with pytest.raises(rx.T41RxError, match="channel out of range"):
            ch.set_map([last + 1, 0])
        for off in offs:
            with pytest.raises(rx.T41RxError, match="aligned"):
                ch.process_device(cap.data_ptr() + off, iq.data_ptr(), 1)
        ch.process_device(cap.data_ptr(), iq.data_ptr(), 1)
        ch.synchronize()
    assert np.all(iq.cpu().numpy() == 0.0)


@pytest.mark.gpu
def test_sideband_at_a_channel_centre_real_1280():
    """A tone 1 kHz above a USB dial at the centre of channel 147 (14.112 MHz) of a 122.88 MS/s capture (M = 1280),
    placed by chan_place_real: 1 kHz audio in USB and >= 65 dB weaker in LSB."""
    M, T = 1280, 8
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
    print("M=1280 USB / LSB %.1f dB" % ratio)
    assert ratio >= 65.0


@pytest.mark.gpu
@pytest.mark.parametrize("M, freq, step", [(1280, 14.140e6, 12), (800, 3.580e6, 16)])
def test_psk31_decodes_real_at_new_rates(M, freq, step):
    """PSK31 on 20 m (14.140 MHz, M = 1280) and on 80 m (3.580 MHz, M = 800), placed by chan_place_real, both 28 kHz
    above their channel's centre; the capture is generated and channelized `step` blocks at a time."""
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
            chan.process_device(cap.data_ptr(), iq[0, b0].data_ptr(), nb)
            chan.synchronize()
    ps = [rx.make_params(mode=rx.DEMOD_USB, f_lo_cut=-100, f_hi_cut=100, agc_mode=0, psk31_enable=1, nco_freq=nco)]
    out = chain(ps, iq.cpu().numpy(), want_psk=True)
    chars = bytes(out["psk_chars"][0][out["psk_chars"][0] > 0])
    assert cases.PSK_TEXT.encode() in chars, chars


@pytest.mark.gpu
def test_bank_placed_by_chan_place_at_640_matches_rotated_reference_feed():
    """32 receivers (USB, LSB, AM, NFM, PSK31-in-USB) across a 61.44 MS/s capture (M = 640), placed by chan_place: the
    chain on the channelizer's output and on the rotated float64 reference rounded to float32 (flags = 0 both): audio
    SNR >= 90 dB after block 2, discrete state identical."""
    M, T, n = 640, 12, 32
    r = np.random.default_rng(34)
    fs = synth.wideband_rate(M)
    signals, params, chmap, shifts = [], [], [], []
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
        ch, shift, nco = rx.chan_place(M, mode, f)
        signals.append(sig)
        chmap.append(ch)
        shifts.append(shift)
        if kind == 4:
            params.append(rx.make_params(mode=mode, f_lo_cut=-100, f_hi_cut=100, agc_mode=0, psk31_enable=1, nco_freq=nco))
        elif kind == 3:
            params.append(rx.make_params(mode=mode, nco_freq=nco, nfm_filter_bw=12000))
        else:
            params.append(rx.make_params(mode=mode, nco_freq=nco))
    capture = synth.wideband(9, M, T, signals, sigma=0.002)
    got_iq = channelize(M, n, capture, [T], [chmap], [shifts])
    x, taps = cplx(capture), rx.chan_taps(M)
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
    print("M=640 bank: worst audio SNR %.1f dB" % worst)
