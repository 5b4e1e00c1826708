"""Channelizer fine tuning (t41rx_chan_set_shift, t41rx_chan_place): each receiver's 192 kS/s stream rotated by its own
frequency, so that a signal anywhere in the capture reaches the chain at NCOFreq 0, where the chain rejects the
opposite sideband best and decodes PSK31.

CPU tier: t41rx_chan_place maps back to every offset of a grid and rejects what t41rx_chan_tune rejects; the placement
rule through the Tier-B oracle chain fed with the float64 channel rotated as the header defines it (sideband rejection
across a channel, the sign for NFM, PSK31 at a channel centre).  GPU tier: the kernel against the float64 formula,
bit-identity of unshifted receivers and across call splits, continuous phase at a shift change, and the chain end to
end on placed receivers.
"""
import numpy as np
import pytest

import cases
import oracle_py as O
from chan_driver import OUT_RATE, chain, channelize, cplx, error_ratio, reference_channel, rotate
from t41_sdr_b200 import rx, synth

CHANNELS = (64, 512)
MIRRORED = (rx.DEMOD_USB, rx.DEMOD_LSB, rx.DEMOD_AM, rx.DEMOD_SAM)
PLAIN = (rx.DEMOD_NFM, rx.DEMOD_PSK31)
BLOCK = rx.BLOCK


def _iq(z, n_blocks):
    return np.stack([z.real, z.imag], -1).astype(np.float32).reshape(n_blocks, BLOCK, 2)


def _mirrored(mode):
    return mode in MIRRORED


# ---------------------------------------------------------------- CPU tier

@pytest.mark.parametrize("M", CHANNELS)
def test_place_maps_back_to_the_offset(M):
    fs = int(synth.wideband_rate(M))
    rng = np.random.default_rng(7 + M)
    offsets = np.concatenate([rng.integers(-fs // 2, fs // 2, 400),
                              [-fs // 2, fs // 2 - 1, 0, 48000, -48000, 47999, 96000, 144000, fs // 2 - 48000,
                               fs // 2 - 48001, -fs // 2 + 48000]])
    for mode in MIRRORED + PLAIN:
        for off in offsets:
            ch, shift, nco = rx.chan_place(M, mode, float(off))
            assert (ch, nco) == (rx.chan_tune(M, mode, float(off))[0], 0)
            f_rel = shift - 48000 if _mirrored(mode) else shift + 48000
            assert abs(f_rel) <= 48000 and abs(shift) < OUT_RATE
            assert (rx.chan_centre(M, ch) + f_rel - int(off)) % fs == 0, (mode, off, ch, shift)


@pytest.mark.parametrize("M", CHANNELS)
def test_place_rejects_what_tune_rejects(M):
    half = synth.wideband_rate(M) / 2
    for off in (half, half + 1, -half - 1, 1e12, float("nan")):
        with pytest.raises(rx.T41RxError, match="t41rx_chan_place"):
            rx.chan_place(M, rx.DEMOD_USB, off)
    for mode in (4, 6, 7, -1, 99):
        with pytest.raises(rx.T41RxError, match="invalid mode"):
            rx.chan_place(M, mode, 0.0)
    with pytest.raises(rx.T41RxError):
        rx.chan_place(128, rx.DEMOD_USB, 0.0)


def _oracle_audio(mode, nco, iq, skip=4, **kw):
    st = O.OracleStream(cases.P(mode=mode, nco_freq=nco, agc_mode=0, **kw))
    try:
        return st.process(iq)["audio"][skip:].ravel().astype(np.float64)
    finally:
        st.close()


def _placed_feed(capture, M, mode, offset, n_blocks):
    """the float64 channel t41rx_chan_place picks for offset, rotated by its shift from m = 0; and its nco_freq"""
    ch, shift, nco = rx.chan_place(M, mode, offset)
    z = reference_channel(cplx(capture), rx.chan_taps(M), M, ch, n_blocks * BLOCK)
    return _iq(rotate(z, 0, shift), n_blocks), nco


@pytest.mark.parametrize("f_rel", [0.0, 20000.0, -20000.0, 47000.0, -47000.0])
def test_placement_rejects_the_opposite_sideband_on_the_oracle(f_rel):
    """A tone 1 kHz above a USB dial placed by chan_place, f_rel from the centre of channel 13: 1 kHz audio in USB,
    >= 70 dB weaker in LSB (chan_tune's placement at f_rel = 0: 19.7 dB)."""
    M, T = 64, 8
    dial = rx.chan_centre(M, 13) + f_rel
    capture = synth.wideband(1, M, T, [("tone", dial + 1000.0, {"amp": 0.1})])
    iq, nco = _placed_feed(capture, M, rx.DEMOD_USB, dial, T)
    assert rx.chan_place(M, rx.DEMOD_LSB, dial) == rx.chan_place(M, rx.DEMOD_USB, dial)
    usb, lsb = _oracle_audio(rx.DEMOD_USB, nco, iq), _oracle_audio(rx.DEMOD_LSB, nco, iq)
    spec = np.abs(np.fft.rfft(usb * np.hanning(usb.size)))
    f_peak = np.argmax(spec) * float(OUT_RATE) / usb.size
    assert abs(f_peak - 1000.0) <= 2 * OUT_RATE / usb.size, f_peak
    ratio = 10 * np.log10(np.mean(usb ** 2) / max(np.mean(lsb ** 2), 1e-300))
    print("f_rel %+.0f: USB / LSB %.1f dB" % (f_rel, ratio))
    assert ratio >= 70.0, ratio


def test_nfm_placement_sign_on_the_oracle():
    """NFM 20 kHz above the centre of channel 13.  A mirrored FM signal demodulates to inverted audio, so a test of the
    tone alone cannot fix the sign of the shift: the placed receiver's audio must correlate with +0.99 or better with
    the same signal fed at chan_tune's placement (no shift).  On the oracle: +0.99995; the opposite shift gives a 1 kHz
    tone too, inverted (-0.65), and the mirrored modes' rule 48000 + f_rel +0.87."""
    M, T = 64, 8
    f = rx.chan_centre(M, 13) + 20000.0
    capture = synth.wideband(2, M, T, [("nfm", f, {"amp": 0.1})])
    ch, nco_direct = rx.chan_tune(M, rx.DEMOD_NFM, f)
    z = reference_channel(cplx(capture), rx.chan_taps(M), M, ch, T * BLOCK)
    direct = _oracle_audio(rx.DEMOD_NFM, nco_direct, _iq(z, T))
    _, shift, nco = rx.chan_place(M, rx.DEMOD_NFM, f)
    assert (shift, nco) == (20000 - 48000, 0)
    placed = _oracle_audio(rx.DEMOD_NFM, nco, _iq(rotate(z, 0, shift), T))
    mirrored = _oracle_audio(rx.DEMOD_NFM, nco, _iq(rotate(z, 0, -shift), T))
    corr = np.corrcoef(direct, placed)[0, 1]
    print("NFM audio RMS direct %.6f placed %.6f, correlation %+.5f (opposite shift %+.5f)"
          % (np.sqrt(np.mean(direct ** 2)), np.sqrt(np.mean(placed ** 2)), corr, np.corrcoef(direct, mirrored)[0, 1]))
    assert corr >= 0.99
    assert np.corrcoef(direct, mirrored)[0, 1] <= -0.5


def _psk_capture(M, offsets, seed=31):
    T = synth.psk31_blocks(cases.PSK_TEXT, 5014)
    signals = [("psk31", f, {"amp": 0.25, "text": cases.PSK_TEXT, "symbol_offset": 5014}) for f in offsets]
    pieces, step = [], 67
    for b0 in range(0, T, step):           # generated piece by piece: the capture is long
        pieces.append(synth.wideband(seed, M, min(step, T - b0), signals, sigma=0.01, start_block=b0))
    return np.concatenate(pieces), T, step


def test_psk31_decodes_at_a_channel_centre_on_the_oracle():
    """PSK31 exactly at the centre of channel 7, placed by chan_place (chan_tune's NCOFreq 48000 does not decode)."""
    M = 64
    f = rx.chan_centre(M, 7)
    capture, T, _ = _psk_capture(M, [f])
    iq, nco = _placed_feed(capture, M, rx.DEMOD_USB, f, T)
    st = O.OracleStream(cases.P(mode=rx.DEMOD_USB, f_lo_cut=-100, f_hi_cut=100, agc_mode=0, psk31_enable=1,
                                nco_freq=nco))
    out = st.process(iq, want_psk=True)
    st.close()
    chars = bytes(out["psk_chars"][out["psk_chars"] > 0])
    assert cases.PSK_TEXT.encode() in chars, chars


# ---------------------------------------------------------------- GPU tier

def _test_capture(M, n_blocks, seed):
    r = np.random.default_rng(seed)
    fs = synth.wideband_rate(M)
    sig = [("tone", float(r.uniform(-fs / 2, fs / 2)), {"amp": float(r.uniform(0.05, 0.5))}) for _ in range(6)]
    sig.append(("tone", rx.chan_centre(M, 7) + 1234.5, {"amp": 0.3}))
    return synth.wideband(seed, M, n_blocks, sig, sigma=0.2)


@pytest.mark.gpu
@pytest.mark.parametrize("M", CHANNELS)
def test_formula_parity_with_shifts(M):
    """Positive, negative, +-96000 and extreme shifts, two receivers on channel 7 with different shifts, an unshifted
    and an unmapped receiver, over two calls: against float64 z_k[m] exp(2 pi j shift m / 192000), error RMS <= 1e-6 of
    the capture's RMS."""
    n_blocks = 4 if M == 64 else 2
    capture = _test_capture(M, n_blocks, 200 + M)
    chmap = [7, 7, 1, M // 2, M - 1, 0, 3, -1, 7]
    shifts = [12345, -54321, 96000, -96000, 191999, -191999, 0, 5000, 48000]
    got = channelize(M, len(chmap), capture, [1, n_blocks - 1], [chmap, None], [shifts, None])
    x, taps = cplx(capture), rx.chan_taps(M)
    want = {r: rotate(reference_channel(x, taps, M, k, n_blocks * BLOCK), 0, s)
            for r, (k, s) in enumerate(zip(chmap, shifts)) if k >= 0}
    assert np.all(got[chmap.index(-1)] == 12345.0)
    ratio = error_ratio(got, want, x)
    print("M=%d: error RMS / capture RMS = %.3g" % (M, ratio))
    assert ratio <= 1e-6


@pytest.mark.gpu
def test_unshifted_receivers_and_split_calls_are_bit_identical():
    """Receivers left at shift 0 give the bits of a channelizer on which set_shift was never called, also on a channel
    shared with a shifted receiver, and so do receivers set to 0 explicitly; with shifts set, 1 + 2 + 5 blocks equal
    one call."""
    M, T = 64, 8
    capture = _test_capture(M, T, 5)
    chmap = [3, 40, 3, 63, 32, 40, -1]
    shifts = [48000, 0, 0, -20000, 0, 95999, 777]
    plain = channelize(M, 7, capture, [T], [chmap])
    one = channelize(M, 7, capture, [T], [chmap], [shifts])
    split = channelize(M, 7, capture, [1, 2, 5], [chmap, None, None], [shifts, None, None])
    zeros = channelize(M, 7, capture, [1, 2, 5], [chmap, None, None], [[0] * 7, None, [0] * 7])
    assert np.array_equal(one.view(np.uint32), split.view(np.uint32))
    assert np.array_equal(zeros.view(np.uint32), plain.view(np.uint32))
    for r, s in enumerate(shifts):
        same = np.array_equal(one[r].view(np.uint32), plain[r].view(np.uint32))
        assert same == (s == 0 or chmap[r] < 0), r


@pytest.mark.gpu
def test_shift_change_keeps_the_phase_continuous():
    """Shifts changed after 3 of 8 blocks (one receiver back to 0, one from 0): against float64 with a piecewise
    frequency and continuous phase, error RMS <= 1e-6 of the capture's RMS."""
    M, T, T1 = 64, 8, 3
    capture = _test_capture(M, T, 11)
    chmap = [7, 7, 20, 50]
    s1 = [30000, -70000, 0, 12345]
    s2 = [-45000, 0, 60000, 12345]
    got = channelize(M, 4, capture, [T1, T - T1], [chmap, None], [s1, s2])
    x, taps = cplx(capture), rx.chan_taps(M)
    m1 = T1 * BLOCK
    want = {}
    for r, k in enumerate(chmap):
        z = reference_channel(x, taps, M, k, T * BLOCK)
        phase1 = (s1[r] * m1) % OUT_RATE                       # where the first shift has brought the phase at m1
        want[r] = np.concatenate([rotate(z[:m1], 0, s1[r]), rotate(z[m1:], phase1, s2[r])])
    ratio = error_ratio(got, want, x)
    print("error RMS / capture RMS = %.3g" % ratio)
    assert ratio <= 1e-6


@pytest.mark.gpu
def test_set_shift_rejects_bad_input():
    with rx.Channelizer(64, 4) as ch:
        for bad in ([192000], [-192000], [0, 0, 0, 10 ** 6]):
            with pytest.raises(rx.T41RxError, match="t41rx_chan_set_shift"):
                ch.set_shift(bad)
        with pytest.raises(rx.T41RxError):
            ch.set_shift([0, 0], first=3)
        with pytest.raises(rx.T41RxError):
            ch.set_shift([0], first=-1)
        ch.set_shift([191999, -191999, 0, 96000])


@pytest.mark.gpu
def test_sideband_at_a_channel_centre_end_to_end():
    """A tone 1 kHz above a USB dial at the centre of channel M - 13, placed by chan_place: 1 kHz audio in USB and
    >= 65 dB weaker in LSB (chan_tune there: NCOFreq 48000, about 20 dB)."""
    M, T = 64, 8
    dial = rx.chan_centre(M, M - 13)
    placed = rx.chan_place(M, rx.DEMOD_USB, dial)
    assert placed == rx.chan_place(M, rx.DEMOD_LSB, dial) == (M - 13, 48000, 0)
    ch, shift, nco = placed
    capture = synth.wideband(1, M, T, [("tone", dial + 1000.0, {"amp": 0.1})])
    iq = channelize(M, 2, capture, [T], [[ch, ch]], [[shift, shift]])
    ps = [rx.make_params(mode=rx.DEMOD_USB, nco_freq=nco, agc_mode=0),
          rx.make_params(mode=rx.DEMOD_LSB, nco_freq=nco, agc_mode=0)]
    audio = chain(ps, iq)["audio"][:, 4:].reshape(2, -1).astype(np.float64)
    spec = np.abs(np.fft.rfft(audio[0] * np.hanning(audio.shape[1])))
    f_peak = np.argmax(spec) * float(OUT_RATE) / audio.shape[1]
    assert abs(f_peak - 1000.0) <= 2 * OUT_RATE / audio.shape[1], f_peak
    ratio = 10 * np.log10(np.mean(audio[0] ** 2) / max(np.mean(audio[1] ** 2), 1e-300))
    print("USB / LSB %.1f dB" % ratio)
    assert ratio >= 65.0


@pytest.mark.gpu
def test_psk31_decodes_at_channel_centres_end_to_end():
    """PSK31 exactly at the centres of channel 7 and channel M - 16 (a negative offset), placed by chan_place."""
    M = 64
    offsets = (rx.chan_centre(M, 7), rx.chan_centre(M, M - 16))
    placed = [rx.chan_place(M, rx.DEMOD_USB, f) for f in offsets]
    assert placed == [(7, 48000, 0), (M - 16, 48000, 0)]
    capture, T, step = _psk_capture(M, offsets)
    calls = [min(step, T - b0) for b0 in range(0, T, step)]
    rest = [None] * (len(calls) - 1)
    iq = channelize(M, 2, capture, calls, [[c for c, _, _ in placed]] + rest, [[s for _, s, _ in placed]] + rest)
    ps = [rx.make_params(mode=rx.DEMOD_USB, f_lo_cut=-100, f_hi_cut=100, agc_mode=0, psk31_enable=1, nco_freq=nco)
          for _, _, nco in placed]
    out = chain(ps, iq, want_psk=True)
    for s in range(2):
        chars = bytes(out["psk_chars"][s][out["psk_chars"][s] > 0])
        assert cases.PSK_TEXT.encode() in chars, (s, chars)


@pytest.mark.gpu
def test_bank_placed_by_chan_place_matches_rotated_reference_feed():
    """The 32-receiver bank of test_bank_fed_by_channelizer_matches_reference_feed, placed by chan_place: the chain on
    the channelizer's output and on the rotated float64 reference rounded to float32 (flags = 0 both): audio SNR
    >= 90 dB after block 2, discrete state identical."""
    M, T, n = 64, 12, 32
    r = np.random.default_rng(32)
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
    ref_iq = np.stack([_iq(rotate(reference_channel(x, taps, M, k, T * BLOCK), 0, s), T)
                       for k, s in zip(chmap, shifts)])
    got, want = chain(params, got_iq), chain(params, ref_iq)
    worst = np.inf
    for s in range(n):
        snr = O.snr_db(want["audio"][s, 2:], got["audio"][s, 2:])
        worst = min(worst, snr)
        assert snr >= 90.0, (s, snr)
        for f in cases.DEBUG_INT_FIELDS:
            assert getattr(got["debug"][s], f) == getattr(want["debug"][s], f), (s, f)
    print("worst audio SNR %.1f dB" % worst)
