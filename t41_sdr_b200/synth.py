"""Deterministic synthetic I/Q for the T41 receive chain (SURVEY.md §8(d), configs C1-C5).

All generators are seeded (seed = 0x74140000 + stream_id), produce float32 arrays
of shape [n_blocks, 2048, 2] (interleaved I,Q per sample, 192 kS/s) and quantise to
the q15 grid (value * 32768 is an integer), which is what the firmware's ADC path
delivers (reference Process.cpp:107-108) and what the Tier-A cross-check requires.

Frequency plan of the chain (reference Process.cpp:165-236): for USB/LSB/AM/SAM the
I channel is negated (spectral mirror), then +Fs/4, then -NCOFreq; NFM/PSK31 skip the
mirror.  `rf_for_baseband` inverts that so a generator can say where a tone should
land after the front end.
"""
import numpy as np

FS = 192000.0
BLOCK = 2048
SEED_BASE = 0x74140000

DEMOD_USB, DEMOD_LSB, DEMOD_AM, DEMOD_NFM, DEMOD_PSK31, DEMOD_SAM = 0, 1, 2, 3, 5, 8
_MIRRORED = (DEMOD_USB, DEMOD_LSB, DEMOD_AM, DEMOD_SAM)


def rng_for(stream_id):
    return np.random.Generator(np.random.PCG64(SEED_BASE + int(stream_id)))


def to_q15_grid(x):
    """Round a float array to the q15 grid and return float32 (x * 32768 integral, |x| < 1)."""
    q = np.clip(np.rint(np.asarray(x, np.float64) * 32768.0), -32768, 32767)
    return (q / 32768.0).astype(np.float32)


def rf_for_baseband(f_baseband, mode, nco_freq=0):
    """Input frequency (Hz, at 192 kS/s) that the front end moves to f_baseband."""
    if mode in _MIRRORED:
        return 48000.0 - nco_freq - f_baseband
    return f_baseband - 48000.0 + nco_freq


def _pack(z):
    n = z.size // BLOCK
    out = np.empty((n, BLOCK, 2), np.float32)
    out[..., 0] = to_q15_grid(z.real).reshape(n, BLOCK)
    out[..., 1] = to_q15_grid(z.imag).reshape(n, BLOCK)
    return out


def _noise(rng, n, sigma):
    return sigma * (rng.standard_normal(n) + 1j * rng.standard_normal(n))


def tone(stream_id, n_blocks, f_baseband=1000.0, mode=DEMOD_USB, nco_freq=0, amp=0.25, sigma=0.01,
         level_step_block=None, level_step_db=0.0):
    """C1: complex tone + white noise, landing at f_baseband after the front end."""
    rng = rng_for(stream_id)
    n = n_blocks * BLOCK
    t = np.arange(n) / FS
    f0 = rf_for_baseband(f_baseband, mode, nco_freq)
    z = amp * np.exp(2j * np.pi * f0 * t)
    z = _apply_step(z, level_step_block, level_step_db) + _noise(rng, n, sigma)
    return _pack(z)


def _apply_step(z, level_step_block, level_step_db):
    if level_step_block is not None:
        g = np.ones(z.size)
        g[level_step_block * BLOCK:] = 10.0 ** (level_step_db / 20.0)
        z = z * g
    return z


def am(stream_id, n_blocks, mode=DEMOD_AM, nco_freq=0, carrier_offset=0.0, depth=0.5, f_mod=400.0,
       amp=0.2, sigma=0.005, level_step_block=None, level_step_db=0.0):
    """C2/C3: AM (or SAM with a small carrier offset) carrier landing at carrier_offset Hz."""
    rng = rng_for(stream_id)
    n = n_blocks * BLOCK
    t = np.arange(n) / FS
    f0 = rf_for_baseband(carrier_offset, mode, nco_freq)
    env = 1.0 + depth * np.sin(2 * np.pi * f_mod * t)
    z = amp * env * np.exp(2j * np.pi * f0 * t)
    z = _apply_step(z, level_step_block, level_step_db) + _noise(rng, n, sigma)
    return _pack(z)


def nfm(stream_id, n_blocks, nco_freq=0, deviation=2500.0, f_mod=1000.0, amp=0.25, sigma=0.005,
        level_step_block=None, level_step_db=0.0):
    """C3: narrow-band FM, carrier landing at 0 Hz."""
    rng = rng_for(stream_id)
    n = n_blocks * BLOCK
    t = np.arange(n) / FS
    f0 = rf_for_baseband(0.0, DEMOD_NFM, nco_freq)
    phase = 2 * np.pi * f0 * t + (deviation / f_mod) * np.sin(2 * np.pi * f_mod * t)
    z = amp * np.exp(1j * phase)
    z = _apply_step(z, level_step_block, level_step_db) + _noise(rng, n, sigma)
    return _pack(z)


def two_tone(stream_id, n_blocks, f1=5000.0, f2=-12000.0, a1=0.2, a2=0.05, sigma=0.01):
    """C4: two raw-input tones (Hz at the 192 kS/s input) + noise for the spectrum rows."""
    rng = rng_for(stream_id)
    n = n_blocks * BLOCK
    t = np.arange(n) / FS
    z = a1 * np.exp(2j * np.pi * f1 * t) + a2 * np.exp(2j * np.pi * f2 * t) + _noise(rng, n, sigma)
    return _pack(z)


# ---- PSK31 (C5) ----
# Varicode alphabet (G3PLX); code words as bit strings, characters separated by "00".
_VARICODE = None


def varicode_table():
    """ascii -> bit string, read from the generated product data header."""
    global _VARICODE
    if _VARICODE is None:
        import os
        import re
        path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "csrc", "rx_tables_data.h")
        txt = open(path).read()
        tab = {}
        for code, bits, asc in re.findall(r"\{0x([0-9a-f]+),\s*(\d+),0x([0-9a-f]+)\}", txt):
            tab[int(asc, 16)] = format(int(code, 16), "0%db" % int(bits))
        assert len(tab) == 128
        _VARICODE = tab
    return _VARICODE


def psk31_bits(text, lead_in=16):
    """Varicode bit stream: idle zeros, then each character followed by '00'."""
    tab = varicode_table()
    bits = [0] * lead_in
    for ch in text.encode("ascii"):
        bits += [int(b) for b in tab[ch]] + [0, 0]
    bits += [0] * 4
    return np.array(bits, np.uint8)


SYMBOL_SAMPLES_192K = 6144  # 31.25 Bd = 768 samples at 24 kS/s = 3 blocks of 2048 at 192 kS/s


def psk31(stream_id, text, nco_freq=0, amp=0.25, ebn0_db=20.0, symbol_offset=0):
    """C5: differentially encoded BPSK31 (bit 0 = phase reversal) with raised-cosine amplitude
    shaping across reversals, carrier landing at 0 Hz.  Symbol centres sit at sample
    symbol_offset + k*6144 + 3072 ... the receiver taps sample 0 of every third decimated
    block, so symbol k is centred `symbol_offset` input samples after the block-3k boundary
    plus the chain's group delay; see tests for the alignment used.
    Returns (iq, bits)."""
    rng = rng_for(stream_id)
    bits = psk31_bits(text)
    n_blocks = psk31_blocks(text, symbol_offset)
    total = n_blocks * BLOCK
    k = np.arange(total) - symbol_offset
    t = np.arange(total) / FS
    f0 = rf_for_baseband(0.0, DEMOD_USB, nco_freq)
    # Eb/N0 at 31.25 Bd referenced to the 192 kS/s complex noise density
    sigma = amp / np.sqrt(2.0 * (10.0 ** (ebn0_db / 10.0)) * 31.25 / FS)
    sigma = min(sigma, 0.2)
    z = amp * _psk31_shape(bits, k) * np.exp(2j * np.pi * f0 * t) + _noise(rng, total, sigma)
    return _pack(z), bits


def _psk31_shape(bits, k):
    """Amplitude of the differentially encoded BPSK31 of `bits` at (possibly fractional) sample k of 192 kS/s, k = 0
    being the start of symbol 0: raised-cosine transitions between the symbol levels, level[0] before the start."""
    n_sym = bits.size
    level = np.empty(n_sym + 1)
    level[0] = 1.0
    for i in range(n_sym):
        level[i + 1] = level[i] * (1.0 if bits[i] else -1.0)
    sps = SYMBOL_SAMPLES_192K
    idx = np.clip(np.floor(k / sps).astype(np.int64), 0, n_sym - 1)
    frac = (k - idx * sps) / float(sps)
    a = level[np.clip(idx, 0, n_sym)]
    b = level[np.clip(idx + 1, 0, n_sym)]
    shape = a + (b - a) * 0.5 * (1.0 - np.cos(np.pi * frac))
    shape[k < 0] = level[0]
    return shape


# ---- wideband captures for the channelizer (t41rx_chan_*) ----
CHAN_SPACING = 96000.0
CHAN_TAPS_PER_BRANCH = 10


def wideband_rate(n_channels):
    """Sample rate of a capture for an n_channels channelizer (Hz)."""
    return n_channels * CHAN_SPACING


def wideband_delay(n_channels):
    """How far (s) a channel lags the capture: the prototype's (N - 1) / 2 samples at the capture rate, that is
    10 - 1 / n_channels output samples."""
    return (CHAN_TAPS_PER_BRANCH * n_channels - 1) / 2.0 / wideband_rate(n_channels)


def psk31_blocks(text, symbol_offset=0):
    """192 kS/s blocks (a multiple of 3) that hold the PSK31 of `text` as psk31() builds it."""
    n = (psk31_bits(text).size + 1) * SYMBOL_SAMPLES_192K
    n_blocks = (n + symbol_offset + BLOCK - 1) // BLOCK
    return ((n_blocks + 2) // 3) * 3


def wideband(seed, n_channels, n_blocks, signals, sigma=0.0, start_block=0):
    """A complex capture at n_channels x 96 kS/s holding n_blocks output blocks' worth of samples (n_blocks * 2048 *
    n_channels / 2), float32 [n, 2] interleaved (I, Q), not quantised.  `signals` is a list of (kind, offset_hz, kw):
      ("tone", f, {amp})                                   exp(2 pi j f t)
      ("am", f, {amp, depth, f_mod})                       carrier at f
      ("nfm", f, {amp, deviation, f_mod})                  carrier at f
      ("psk31", f, {amp, text, symbol_offset})             BPSK31 carrier at f
    f is relative to the capture's centre.  Envelopes are closed-form in t, evaluated at the capture rate.  PSK31 is
    timed in the channel's clock: symbol k is centred at output sample symbol_offset + 6144 k + 3072 of the channel,
    as psk31() centres it in its own stream, so a receiver decodes it with the same alignment.  start_block shifts t
    (a later piece of the same capture); the noise (sigma per component) comes from seed and start_block."""
    z = _wideband_sum(seed, n_channels, n_blocks, signals, sigma, start_block)
    out = np.empty((z.size, 2), np.float32)
    out[:, 0] = z.real
    out[:, 1] = z.imag
    return out


def wideband_real(seed, n_channels, n_blocks, signals, sigma=0.0, start_block=0):
    """A real capture at n_channels x 96 kS/s (n_channels 128, 800, 1024 or 1280) as a direct-sampling ADC delivers
    it: int16 round(32768 Re z), saturated, n_blocks * 2048 * n_channels / 2 samples.  z is the sum wideband() forms
    with the same arguments, f measured from 0 Hz, so a ("tone", f, {amp}) is amp cos(2 pi f t)."""
    z = _wideband_sum(seed, n_channels, n_blocks, signals, sigma, start_block)
    return np.clip(np.round(32768.0 * z.real), -32768, 32767).astype(np.int16)


def wideband_q15(seed, n_channels, n_blocks, signals, sigma=0.0, start_block=0):
    """A complex capture at n_channels x 96 kS/s (n_channels 64, 320, 512 or 640) as a wideband I/Q digitizer streams
    it (sc16): int16 [n, 2] interleaved (I, Q), round(32768 z) saturated to [-32768, 32767] per component.  z is the
    sum wideband() forms with the same arguments, so wideband_q15 / 32768 is wideband() quantised."""
    z = _wideband_sum(seed, n_channels, n_blocks, signals, sigma, start_block)
    out = np.empty((z.size, 2), np.int16)
    out[:, 0] = np.clip(np.round(32768.0 * z.real), -32768, 32767)
    out[:, 1] = np.clip(np.round(32768.0 * z.imag), -32768, 32767)
    return out


def _wideband_sum(seed, n_channels, n_blocks, signals, sigma, start_block):
    """complex128 signal sum and noise of wideband() / wideband_real() / wideband_q15()"""
    fs = wideband_rate(n_channels)
    per_block = BLOCK * n_channels // 2
    n = n_blocks * per_block
    n0 = start_block * per_block
    t = (n0 + np.arange(n)) / fs
    z = np.zeros(n, np.complex128)
    for kind, f, kw in signals:
        carrier = np.exp(2j * np.pi * ((f * (n0 + np.arange(n))) % fs) / fs)   # phase reduced exactly for large n
        if kind == "tone":
            z += kw.get("amp", 0.25) * carrier
        elif kind == "am":
            env = 1.0 + kw.get("depth", 0.5) * np.sin(2 * np.pi * kw.get("f_mod", 400.0) * t)
            z += kw.get("amp", 0.2) * env * carrier
        elif kind == "nfm":
            dev, fm = kw.get("deviation", 2500.0), kw.get("f_mod", 1000.0)
            z += kw.get("amp", 0.25) * carrier * np.exp(1j * (dev / fm) * np.sin(2 * np.pi * fm * t))
        elif kind == "psk31":
            bits = psk31_bits(kw["text"])
            k = (t + wideband_delay(n_channels)) * FS - kw.get("symbol_offset", 0)
            z += kw.get("amp", 0.25) * _psk31_shape(bits, k) * carrier
        else:
            raise ValueError("unknown signal kind %r" % (kind,))
    if sigma > 0.0:
        z += _noise(np.random.Generator(np.random.PCG64([SEED_BASE + int(seed), int(start_block)])), n, sigma)
    return z
