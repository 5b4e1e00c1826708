"""Diversity channelizer (DESIGN §3.11): n_inputs = 2 ... 4 coherent captures of one kind, receiver r mapped to channel k
getting rot_r(m) sum_a w[r][a] z^(a)_k[m], z^(a)_k being the single-input channelizer's channel of input a.

CPU tier: argument checks at creation (every kind), ENODEV without a device, the Python binding's n_inputs check, the
synth helpers' coherence, and the weight convention in float64: sum_a w_a z(x_a) is the channel of the combined capture
sum_a conj(w_a) x_a (the channelizer's conjugate).

GPU tier, at every (kind, M) of the twelve kernel instances: default weights give the single-input channelizer's bits;
seeded weights against float64 (error RMS / (sum_a |w_a| RMS(x_a)) <= 2e-7: the single-input bound 1e-7 plus one
complex product and one sum); call splits and a weight change between calls; a null against the float64 model's; four
inputs on one M per kind; the chain end to end on nulled and un-nulled receivers.
"""
import ctypes as C

import numpy as np
import pytest

import cases
import oracle_py as O
from chan_driver import chain, channelize, cplx, reference_all_channels
from t41_sdr_b200 import rx, synth

BLOCK = rx.BLOCK
OUT_RATE = 192000
EINVAL, ENODEV = -1, -4
FILL = 12345.0
COMPLEX = (64, 320, 512, 640)
REAL = (128, 800, 1024, 1280)
KINDS = [("float", m) for m in COMPLEX] + [("q15", m) for m in COMPLEX] + [("real", m) for m in REAL]
KIND_CODE = {"float": rx.CHAN_FLOAT, "q15": rx.CHAN_Q15, "real": rx.CHAN_REAL}
BOUND = 2e-7                # error RMS / (sum_a |w_a| RMS(x_a)), per receiver
FOUR_INPUTS = [("float", 320), ("q15", 64), ("real", 800)]


def _opts(kind):
    return {"real": kind == "real", "q15": kind == "q15"}


def _n_channels(kind, M):
    return M // 2 + 1 if kind == "real" else M


def _centre(kind, M, k):
    return rx.chan_centre_real(k) if kind == "real" else rx.chan_centre(M, k)


def _x(kind, capture):
    """the capture as the channelizer reads it, complex128"""
    if kind == "real":
        return capture.astype(np.float64) / 32768.0
    return cplx(capture) / (32768.0 if kind == "q15" else 1.0)


def _rms(x):
    return float(np.sqrt(np.mean(np.abs(x) ** 2)))


def _as_complex(iq):
    z = iq[..., 0].astype(np.float64) + 1j * iq[..., 1].astype(np.float64)
    return z.reshape(z.shape[:-2] + (-1,))


def _bits_equal(a, b):
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


def _rotor(shift, m):
    """exp(2 pi j (shift m mod 192000) / 192000) for receivers' shifts [R] and outputs m [n] (counted from creation)"""
    phi = (np.asarray(shift, np.int64)[:, None] * np.asarray(m, np.int64)[None, :]) % OUT_RATE
    return np.exp(2j * np.pi * phi / OUT_RATE)


def _captures(kind, M, n_blocks, n_inputs, seed):
    """n_inputs different seeded captures of the kind (tones and noise, each its own), so that every input's channels
    carry something of their own"""
    r = np.random.default_rng(seed)
    fs = synth.wideband_rate(M)
    lo = 0.0 if kind == "real" else -fs / 2
    out = []
    for a in range(n_inputs):
        sig = [("tone", float(r.uniform(lo, fs / 2)), {"amp": float(r.uniform(0.03, 0.15))}) for _ in range(5)]
        gen = {"float": synth.wideband, "q15": synth.wideband_q15, "real": synth.wideband_real}[kind]
        out.append(gen(seed * 10 + a, M, n_blocks, sig, sigma=0.05))
    return out


def _weights(r, n_recv, n_inputs):
    """seeded complex weights [n_recv, n_inputs]: random (0.1 <= |w| <= 2), and among them 0, 1, -1, -8, 8 j and
    8 exp(j 2.1); no receiver has all weights 0"""
    w = r.uniform(0.1, 2.0, (n_recv, n_inputs)) * np.exp(2j * np.pi * r.uniform(0, 1, (n_recv, n_inputs)))
    special = np.array([0, 1, -1, -8, 8j, 8 * np.exp(2.1j)])
    pick = r.random((n_recv, n_inputs)) < 0.4
    w[pick] = special[r.integers(0, special.size, int(pick.sum()))]
    w[np.all(w == 0, axis=1), 0] = 1.0
    return w


def channelize_diversity(M, n_recv, captures, calls, maps, shifts=None, weights=None, fill=FILL, **kind):
    """chan_driver.channelize() for a diversity channelizer on the coherent `captures` (list, input 0 first):
    weights[i] (None or a complex [count, n_inputs] array for receivers 0 ...) is set before call i, after maps[i] and
    shifts[i].  Returns host iq [n_recv, sum(calls), 2048, 2]; rows of unmapped receivers keep `fill`."""
    import torch
    shifts = shifts or [None] * len(calls)
    weights = weights or [None] * len(calls)
    per_block = BLOCK * M // 2
    d_caps = [torch.from_numpy(np.ascontiguousarray(c)).cuda() for c in captures]
    outs = []
    with rx.Channelizer(M, n_recv, n_inputs=len(captures), **kind) as ch:
        b0 = 0
        for nb, chmap, sh, w in zip(calls, maps, shifts, weights):
            if chmap is not None:
                ch.set_map(chmap)
            if sh is not None:
                ch.set_shift(sh)
            if w is not None:
                ch.set_weights(w)
            d_iq = torch.full((n_recv, nb, BLOCK, 2), fill, dtype=torch.float32, device="cuda")
            ch.process_device([d[b0 * per_block:(b0 + nb) * per_block].data_ptr() for d in d_caps], d_iq.data_ptr(), nb)
            ch.synchronize()
            outs.append(d_iq.cpu().numpy())
            b0 += nb
    return np.concatenate(outs, axis=1)


def _every_channel_case(kind, M, seed):
    """receivers 0 .. n_ch-1 on channels 0 .. n_ch-1 unshifted, n_ch .. 2 n_ch-1 on the same channels with seeded
    shifts (+-1, +-96000 and +-191999 among them), one unmapped receiver last"""
    n_ch = _n_channels(kind, M)
    r = np.random.default_rng(seed)
    shifts = r.integers(-OUT_RATE + 1, OUT_RATE, n_ch)
    special = [1, -1, 96000, -96000, 191999, -191999]
    shifts[r.choice(n_ch, len(special), replace=False)] = special
    return list(range(n_ch)) * 2 + [-1], [0] * n_ch + [int(s) for s in shifts] + [777]


# ---------------------------------------------------------------- CPU tier

@pytest.mark.parametrize("kind", ["float", "q15", "real"])
def test_create_diversity_rejects_bad_arguments(kind):
    """EINVAL, before any device is looked for: an M the kind does not take, n_inputs outside 2 ... 4, n_receivers <= 0"""
    h = C.c_void_p()
    L = rx.lib()
    good_m = 1024 if kind == "real" else 512
    for m in ((320, 640, 512, 64, 100) if kind == "real" else (128, 800, 1024, 1280, 100)):
        assert L.t41rx_chan_create_diversity(C.byref(h), KIND_CODE[kind], m, 2, 4, 0) == EINVAL
        assert b"n_channels must be" in L.t41rx_last_error()
    for n_in in (-1, 0, 1, 5, 8):
        assert L.t41rx_chan_create_diversity(C.byref(h), KIND_CODE[kind], good_m, n_in, 4, 0) == EINVAL
        assert b"n_inputs must be 2, 3 or 4" in L.t41rx_last_error()
    assert L.t41rx_chan_create_diversity(C.byref(h), KIND_CODE[kind], good_m, 2, 0, 0) == EINVAL
    assert L.t41rx_chan_create_diversity(None, KIND_CODE[kind], good_m, 2, 4, 0) == EINVAL
    assert not h.value


def test_create_diversity_rejects_an_unknown_kind():
    h = C.c_void_p()
    for kind in (-1, 3, 7):
        assert rx.lib().t41rx_chan_create_diversity(C.byref(h), kind, 512, 2, 4, 0) == EINVAL
        assert b"kind must be" in rx.lib().t41rx_last_error()
    assert not h.value


def test_weights_and_diversity_call_reject_a_null_channelizer():
    L = rx.lib()
    w = (C.c_float * 4)(1, 0, 0, 0)
    assert L.t41rx_chan_set_weights(None, 0, 1, w) == EINVAL
    caps = (C.c_void_p * 2)(16, 32)
    assert L.t41rx_chan_process_device_diversity(None, caps, C.c_void_p(64), 1, None) == EINVAL


@pytest.mark.parametrize("kind, M", [("float", 512), ("q15", 640), ("real", 1280)])
def test_create_diversity_without_device_is_enodev(kind, M):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    h = C.c_void_p()
    assert rx.lib().t41rx_chan_create_diversity(C.byref(h), KIND_CODE[kind], M, 2, 4, 0) == ENODEV
    assert b"no CUDA device" in rx.lib().t41rx_last_error()
    assert not h.value


@pytest.mark.parametrize("n_inputs", [0, 5, -1, 2.0])
def test_channelizer_rejects_n_inputs_outside_1_to_4(n_inputs):
    with pytest.raises(ValueError):
        rx.Channelizer(512, 4, n_inputs=n_inputs)


def test_synth_diversity_captures_are_coherent():
    """with noise off and no wanted signal, input 1 is exactly c times input 0 (complex sums), the float captures are
    those sums rounded to float32, the sc16 ones quantised as wideband_q15; a real input 1 is g times input 0 delayed by
    d samples, exactly, and the int16 captures are its rounding; noise is independent per input"""
    M, T, c = 64, 2, 0.6 * np.exp(0.7j)
    interf = [("tone", 1.234e6, {"amp": 0.2}), ("am", -0.5e6, {"amp": 0.1})]
    wanted = [("tone", 2.0e6, {"amp": 0.01})]
    z = synth.diversity_sums(3, M, T, [], interf, [1.0, c])
    assert np.array_equal(z[1], c * z[0])
    f = synth.wideband_diversity(3, M, T, [], interf, [1.0, c])
    for a in range(2):
        assert np.array_equal(f[a][:, 0], z[a].real.astype(np.float32))
        assert np.array_equal(f[a][:, 1], z[a].imag.astype(np.float32))
    q = synth.wideband_diversity_q15(3, M, T, [], interf, [1.0, c])
    for a in range(2):
        assert np.array_equal(q[a][:, 0], np.clip(np.round(32768.0 * z[a].real), -32768, 32767).astype(np.int16))
        assert np.array_equal(q[a][:, 1], np.clip(np.round(32768.0 * z[a].imag), -32768, 32767).astype(np.int16))
    Mr, g, d = 128, -0.7, 37
    zr = synth.diversity_sums(4, Mr, T, [], [("tone", 3.21e6, {"amp": 0.3})], [1.0, g], delays=[0, d])
    assert np.array_equal(zr[1][d:], g * zr[0][:-d])
    qr = synth.wideband_diversity_real(4, Mr, T, [], [("tone", 3.21e6, {"amp": 0.3})], [1.0, g], [0, d])
    assert np.array_equal(qr[1], np.clip(np.round(32768.0 * zr[1].real), -32768, 32767).astype(np.int16))
    # the wanted signal goes to input 0 only; noise differs between inputs
    zw = synth.diversity_sums(3, M, T, wanted, interf, [1.0, c])
    assert np.array_equal(zw[1], z[1]) and not np.array_equal(zw[0], z[0])
    zn = synth.diversity_sums(3, M, T, [], [], [1.0, 1.0], sigma=0.01)
    assert abs(np.vdot(zn[0], zn[1])) < 0.05 * np.vdot(zn[0], zn[0]).real


@pytest.mark.parametrize("M", [64, 320])
def test_weight_convention_in_float64(M):
    """the weights multiply the channel as delivered, after the conjugate: sum_a w_a z(x_a) equals z of the combined
    capture sum_a conj(w_a) x_a (max difference <= 1e-12 of the channel RMS); so an input-1 copy c x of x is nulled by
    w1 = -w0 / conj(c)"""
    n_out = 64
    r = np.random.default_rng(M)
    n = n_out * M // 2
    xs = [r.standard_normal(n) + 1j * r.standard_normal(n) for _ in range(3)]
    w = np.array([0.8 - 0.3j, -1.7 + 0.2j, 0.05j])
    taps = rx.chan_taps(M)
    lhs = sum(w[a] * reference_all_channels(xs[a], taps, M, n_out) for a in range(3))
    rhs = reference_all_channels(sum(np.conj(w[a]) * xs[a] for a in range(3)), taps, M, n_out)
    assert np.max(np.abs(lhs - rhs)) <= 1e-12 * _rms(rhs)
    c = 0.4 * np.exp(-1.1j)
    null = reference_all_channels(xs[0], taps, M, n_out) - (1 / np.conj(c)) * reference_all_channels(c * xs[0], taps, M, n_out)
    assert np.max(np.abs(null)) <= 1e-12 * _rms(rhs)


# ---------------------------------------------------------------- GPU tier

def _default_weights_case(kind, M, n_inputs):
    T, calls = 3, [1, 2]
    n_ch = _n_channels(kind, M)
    chmap, shifts = _every_channel_case(kind, M, 900 + M + len(kind))
    n_recv = len(chmap)
    caps = _captures(kind, M, T, n_inputs, 40 + M)
    got = channelize_diversity(M, n_recv, caps, calls, [chmap, None], [shifts, None], fill=FILL, **_opts(kind))
    want = channelize(M, n_recv, caps[0], calls, [chmap, None], [shifts, None], fill=FILL, **_opts(kind))
    assert np.all(got[-1] == FILL)
    assert _bits_equal(got, want)
    # the same, with the default weights set explicitly after a call with other weights
    w = np.zeros((n_recv, n_inputs), np.complex128)
    w[:, 0] = 1.0
    w_other = w.copy()
    w_other[:, -1] = 0.5j
    got2 = channelize_diversity(M, n_recv, caps, calls, [chmap, None], [shifts, None], [w_other, w], fill=FILL,
                                **_opts(kind))
    assert _bits_equal(got2[:, 1:], want[:, 1:])
    print("%s M=%d, %d inputs, default weights: %d receivers bit-identical to the single-input channelizer" % (
        kind, M, n_inputs, n_ch * 2))


@pytest.mark.gpu
@pytest.mark.parametrize("kind, M", KINDS)
def test_default_weights_give_the_single_input_bits(kind, M):
    """2 inputs, default weights (and the defaults set again after a call with other weights): iq bit for bit that of
    the single-input channelizer of the kind on input 0, every channel unshifted and with seeded shifts (+-96000 and
    +-191999 among them); the unmapped receiver keeps its fill"""
    _default_weights_case(kind, M, 2)


def _accuracy_case(kind, M, n_inputs):
    T, calls = 3, [1, 2]
    n_ch = _n_channels(kind, M)
    chmap, shifts = _every_channel_case(kind, M, 700 + M + len(kind))
    n_recv = len(chmap)
    caps = _captures(kind, M, T, n_inputs, 60 + M)
    w = _weights(np.random.default_rng(M + 7 * n_inputs), n_recv, n_inputs)
    got = channelize_diversity(M, n_recv, caps, calls, [chmap, None], [shifts, None], [w, None], fill=FILL,
                               **_opts(kind))
    assert np.all(got[-1] == FILL)
    taps, m = rx.chan_taps(M), np.arange(T * BLOCK)
    xs = [_x(kind, c) for c in caps]
    zs = [reference_all_channels(x, taps, M, T * BLOCK)[:n_ch] for x in xs]
    rot = np.concatenate([np.ones((n_ch, T * BLOCK)), _rotor(shifts[n_ch:-1], m)])
    k = np.array(chmap[:-1])
    want = rot * sum(w[:-1, a, None] * zs[a][k] for a in range(n_inputs))
    err = _as_complex(got[:-1]) - want
    scale = sum(np.abs(w[:-1, a]) * _rms(xs[a]) for a in range(n_inputs))
    ratio = np.sqrt(np.mean(np.abs(err) ** 2, axis=1)) / scale
    r_worst = int(np.argmax(ratio))
    print("%s M=%d, %d inputs: worst error RMS / (sum |w| RMS(x)) %.3g (channel %d, shift %d, w %s), median %.3g" % (
        kind, M, n_inputs, ratio[r_worst], chmap[r_worst], shifts[r_worst], np.round(w[r_worst], 3), np.median(ratio)))
    assert ratio.max() <= BOUND, (chmap[r_worst], shifts[r_worst], w[r_worst], ratio[r_worst])


@pytest.mark.gpu
@pytest.mark.parametrize("kind, M", KINDS)
def test_weighted_channels_against_float64(kind, M):
    """2 inputs, seeded weights on every channel (0, 1, -1, |w| = 8 and random ones), unshifted and shifted: per
    receiver error RMS / (sum_a |w_a| RMS(x_a)) <= 2e-7 against rot * sum_a w_a z^(a) in float64"""
    _accuracy_case(kind, M, 2)


@pytest.mark.gpu
@pytest.mark.parametrize("kind, M", FOUR_INPUTS)
def test_four_inputs(kind, M):
    """n_inputs = 4: default weights give the single-input bits, seeded weights pass the float64 bound"""
    _default_weights_case(kind, M, 4)
    _accuracy_case(kind, M, 4)


@pytest.mark.gpu
@pytest.mark.parametrize("kind, M", KINDS)
def test_call_splits_and_weight_changes(kind, M):
    """one 8-block call is bit-identical to 1 + 2 + 5 block calls (shifted receivers, seeded weights); weights changed
    between calls of 1 + 2 blocks take effect in a step at the boundary: the float64 reference with the old weights
    before it and the new ones after it, within the bound"""
    n_ch = _n_channels(kind, M)
    r = np.random.default_rng(M + 3)
    n_recv = 12
    chmap = [int(v) for v in r.integers(0, n_ch, n_recv)]
    chmap[0] = chmap[1]
    shifts = [int(v) for v in r.integers(-OUT_RATE + 1, OUT_RATE, n_recv)]
    shifts[2] = 0
    w0, w1 = _weights(r, n_recv, 2), _weights(r, n_recv, 2)
    caps = _captures(kind, M, 8, 2, 20 + M)
    one = channelize_diversity(M, n_recv, caps, [8], [chmap], [shifts], [w0], **_opts(kind))
    split = channelize_diversity(M, n_recv, caps, [1, 2, 5], [chmap, None, None], [shifts, None, None],
                                 [w0, None, None], **_opts(kind))
    assert _bits_equal(one, split)
    T = 3
    per_block = BLOCK * M // 2
    head = [c[:T * per_block] for c in caps]
    got = channelize_diversity(M, n_recv, head, [1, 2], [chmap, None], [shifts, None], [w0, w1], **_opts(kind))
    taps = rx.chan_taps(M)
    xs = [_x(kind, c) for c in head]
    zs = [reference_all_channels(x, taps, M, T * BLOCK)[chmap] for x in xs]
    m = np.arange(T * BLOCK)
    wt = np.where(m[None, None, :] < BLOCK, w0[:, :, None], w1[:, :, None])     # [recv, input, m]
    want = _rotor(shifts, m) * sum(wt[:, a] * zs[a] for a in range(2))
    err = _as_complex(got) - want
    scale = sum(np.maximum(np.abs(w0[:, a]), np.abs(w1[:, a])) * _rms(xs[a]) for a in range(2))
    ratio = np.sqrt(np.mean(np.abs(err) ** 2, axis=1)) / scale
    print("%s M=%d weight change: worst error ratio %.3g" % (kind, M, ratio.max()))
    assert ratio.max() <= BOUND, ratio


def _tone_coef(z, f_ch, m0=BLOCK):
    """complex amplitude of exp(2 pi j f_ch m / 192000) in z[m0:] (f_ch a multiple of 192000 / len: exact bins)"""
    m = np.arange(m0, z.shape[-1])
    return np.mean(z[..., m0:] * np.exp(-2j * np.pi * f_ch * m / OUT_RATE), axis=-1)


def _null_case(kind, M, T=4):
    """the captures, channel, weights and float64 model of test_null_matches_the_float64_model"""
    n_ch = _n_channels(kind, M)
    k = n_ch // 3
    ck = _centre(kind, M, k)
    # the conjugate puts capture offset f - c_k at -(f - c_k) in the channel; both on 31.25 Hz bins of T - 1 blocks
    df_i, df_w = -12500.0, 5000.0
    interf = [("tone", ck + df_i, {"amp": 0.3})]
    wanted = [("tone", ck + df_w, {"amp": 0.05})]
    sigma = 0.002 * np.sqrt(M / 64)          # noise that bounds the null near 85 dB at every M
    taps = rx.chan_taps(M)
    if kind == "real":
        g, d = -0.55, 37
        caps = synth.wideband_diversity_real(5, M, T, wanted, interf, [1.0, g], [0, d], sigma=sigma)
        clean = synth.diversity_sums(5, M, T, [], interf, [1.0, g], delays=[0, d])
        zc = [reference_all_channels(z.real, taps, M, T * BLOCK)[k] for z in clean]
        w1 = -_tone_coef(zc[0], -df_i) / _tone_coef(zc[1], -df_i)
    else:
        c = 0.55 * np.exp(1.9j)
        gen = synth.wideband_diversity_q15 if kind == "q15" else synth.wideband_diversity
        caps = gen(5, M, T, wanted, interf, [1.0, c], sigma=sigma)
        w1 = -1.0 / np.conj(c)
    z = [reference_all_channels(_x(kind, cap), taps, M, T * BLOCK)[k] for cap in caps]
    return caps, k, -df_i, -df_w, w1, [z[0], z[0] + w1 * z[1]]


@pytest.mark.gpu
@pytest.mark.parametrize("kind, M", KINDS)
def test_null_matches_the_float64_model(kind, M):
    """An interferer on both inputs (complex: input 1 = c times it; real: gain g, 37 samples later), a wanted tone on
    input 0 only and independent noise per input, in one channel.  Receiver 0 un-nulled (default weights), receiver 1
    nulled: w1 = -1 / conj(c) (complex) or minus the ratio of the interferer's two channels in the float64 reference
    (real, the delayed copy).  The float64 model's null on the same quantised captures is >= 60 dB (the noise bounds
    it); the GPU's is within 1 dB of it; the wanted tone's level in the nulled receiver is within 0.01 dB of the
    un-nulled one's"""
    caps, k, f_i, f_w, w1, model = _null_case(kind, M)
    got = _as_complex(channelize_diversity(M, 2, caps, [4], [[k, k]], None, [np.array([[1.0, 0.0], [1.0, w1]])],
                                           **_opts(kind)))
    i_model = [abs(_tone_coef(v, f_i)) for v in model]
    i_got = [abs(_tone_coef(v, f_i)) for v in got]
    null_model = 20 * np.log10(i_model[0] / i_model[1])
    null_got = 20 * np.log10(i_got[0] / i_got[1])
    wanted_db = 20 * np.log10(abs(_tone_coef(got[1], f_w)) / abs(_tone_coef(got[0], f_w)))
    print("%s M=%d: null %.2f dB (float64 model %.2f dB), wanted tone nulled / un-nulled %+.4f dB" % (
        kind, M, null_got, null_model, wanted_db))
    assert null_model >= 60.0
    assert abs(null_got - null_model) <= 1.0
    assert abs(wanted_db) <= 0.01


def _debug_ints(d):
    return [getattr(d, f) for f in cases.DEBUG_INT_FIELDS]


@pytest.mark.gpu
def test_nulled_usb_receiver_through_the_chain_real_1280():
    """Two ADCs at 122.88 MS/s (M = 1280): a weak USB signal (1 kHz above a 14.2 MHz dial) on ADC 0 only, a strong
    interferer 1.7 kHz above the dial on both (ADC 1: gain -0.8, 23 samples later).  Two USB receivers placed by
    chan_place_real: default weights, and nulling (w1 from the float64 reference's channel ratio at the interferer).
    The nulled receiver's audio against the chain fed with the float64 reference of its combined, rotated channel:
    audio SNR >= 90 dB after block 2, discrete state identical; the interferer's audio tone >= 40 dB below the un-nulled
    receiver's, the wanted tone within 0.5 dB"""
    M, T = 1280, 12
    dial = 14.2e6
    ch, shift, nco = rx.chan_place_real(M, rx.DEMOD_USB, dial)
    wanted = [("tone", dial + 1000.0, {"amp": 0.002})]
    interf = [("tone", dial + 1700.0, {"amp": 0.2})]
    caps = synth.wideband_diversity_real(8, M, T, wanted, interf, [1.0, -0.8], [0, 23], sigma=1e-5)
    taps = rx.chan_taps(M)
    z = [reference_all_channels(x, taps, M, T * BLOCK)[ch] for x in (_x("real", c) for c in caps)]
    f_ch = -(dial + 1700.0 - rx.chan_centre_real(ch))       # the interferer in the channel (31.25 Hz bins)
    w1 = -_tone_coef(z[0], f_ch) / _tone_coef(z[1], f_ch)
    w = np.array([[1.0, 0.0], [1.0, w1]])
    got_iq = channelize_diversity(M, 2, caps, [T], [[ch, ch]], [[shift, shift]], [w], real=True)
    ref = _rotor([shift], np.arange(T * BLOCK))[0] * (z[0] + w1 * z[1])
    ref_iq = np.empty((1, T, BLOCK, 2), np.float32)
    ref_iq[0, ..., 0] = ref.real.reshape(T, BLOCK)
    ref_iq[0, ..., 1] = ref.imag.reshape(T, BLOCK)
    ps = [rx.make_params(mode=rx.DEMOD_USB, nco_freq=nco, agc_mode=0)] * 2
    got = chain(ps, got_iq)
    want = chain(ps[:1], ref_iq)
    snr = O.snr_db(want["audio"][0, 2:], got["audio"][1, 2:])
    assert _debug_ints(got["debug"][1]) == _debug_ints(want["debug"][0])
    audio = got["audio"][:, 4:].reshape(2, -1).astype(np.float64)
    t = np.arange(audio.shape[1]) / 192000.0
    win = np.hanning(audio.shape[1])

    def level(x, f):
        return abs(np.sum(win * x * np.exp(-2j * np.pi * f * t)))

    interf_db = 20 * np.log10(level(audio[0], 1700.0) / level(audio[1], 1700.0))
    wanted_db = 20 * np.log10(level(audio[1], 1000.0) / level(audio[0], 1000.0))
    print("real 1280 through the chain: nulled receiver audio SNR %.1f dB, interferer %.1f dB down, wanted %+.3f dB" % (
        snr, interf_db, wanted_db))
    assert snr >= 90.0
    assert interf_db >= 40.0
    assert abs(wanted_db) <= 0.5


@pytest.mark.gpu
def test_weighted_bank_at_640_q15_matches_combined_reference_feed():
    """32 receivers (USB, LSB, AM, NFM, PSK31-in-USB) across two coherent sc16 captures at 61.44 MS/s (M = 640), placed
    by chan_place, each with its own weights (some nulling an interferer present on both inputs, some random), against
    the chain fed with the float64 reference of each receiver's combined, rotated channel: audio SNR >= 90 dB after
    block 2, discrete state identical.  (12 blocks are too few for a PSK31 message: the next test decodes one.)"""
    M, T, n = 640, 12, 32
    r = np.random.default_rng(35)
    fs = synth.wideband_rate(M)
    c = 0.7 * np.exp(-2.3j)
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
    interf = [("tone", float(r.uniform(-fs / 2, fs / 2)), {"amp": 0.05}) for _ in range(8)]
    caps = synth.wideband_diversity_q15(9, M, T, signals, interf, [1.0, c], sigma=0.002)
    w = np.ones((n, 2), np.complex128)
    w[:, 1] = 0.3 * r.uniform(0, 1, n) * np.exp(2j * np.pi * r.uniform(0, 1, n))
    w[0::3, 1] = -1.0 / np.conj(c)
    w[1::7, 0] = 0.5 - 0.5j
    got_iq = channelize_diversity(M, n, caps, [T], [chmap], [shifts], [w], q15=True)
    taps = rx.chan_taps(M)
    zs = [reference_all_channels(_x("q15", cap), taps, M, T * BLOCK)[chmap] for cap in caps]
    ref = _rotor(shifts, np.arange(T * BLOCK)) * (w[:, 0, None] * zs[0] + w[:, 1, None] * zs[1])
    ref_iq = np.empty_like(got_iq)
    ref_iq[..., 0] = ref.real.reshape(n, T, BLOCK)
    ref_iq[..., 1] = ref.imag.reshape(n, T, BLOCK)
    got, want = chain(params, got_iq), chain(params, ref_iq)
    worst = np.inf
    for s in range(n):
        snr = O.snr_db(want["audio"][s, 2:], got["audio"][s, 2:])
        worst = min(worst, snr)
        assert snr >= 90.0, (s, snr)
        assert _debug_ints(got["debug"][s]) == _debug_ints(want["debug"][s]), s
    print("q15 M=640 weighted bank: worst audio SNR %.1f dB" % worst)


@pytest.mark.gpu
def test_psk31_decodes_through_weighted_receivers_q15_640():
    """Two PSK31 signals across two coherent sc16 captures at 61.44 MS/s (M = 640), on input 0 only, at the centres of
    channels 101 and 407; an interferer 40 Hz above the first carrier, twice its amplitude, on both inputs (input 1:
    c times it).  Receiver 0, placed by chan_place on the first, nulls it (w1 = -1 / conj(c)); receiver 1, on the
    second, has arbitrary weights (input 1 adds only its noise there).  Both decode the message; the captures are
    generated and channelized 24 blocks at a time"""
    import torch
    M, step, text = 640, 24, "CQ DIV"
    T = synth.psk31_blocks(text, 5014)
    c = 0.7 * np.exp(-2.3j)
    f = [rx.chan_centre(M, 101), rx.chan_centre(M, 407)]
    signals = [("psk31", fk, {"amp": 0.1, "text": text, "symbol_offset": 5014}) for fk in f]
    interf = [("tone", f[0] + 40.0, {"amp": 0.2})]
    placed = [rx.chan_place(M, rx.DEMOD_USB, fk) for fk in f]
    w = np.array([[1.0, -1.0 / np.conj(c)], [0.8 + 0.3j, 0.2 - 0.1j]])
    iq = np.empty((2, T, BLOCK, 2), np.float32)
    with rx.Channelizer(M, 2, q15=True, n_inputs=2) as chan:
        chan.set_map([p[0] for p in placed])
        chan.set_shift([p[1] for p in placed])
        chan.set_weights(w)
        for b0 in range(0, T, step):
            nb = min(step, T - b0)
            caps = [torch.from_numpy(cap).cuda() for cap in
                    synth.wideband_diversity_q15(31, M, nb, signals, interf, [1.0, c], sigma=0.002, start_block=b0)]
            d_iq = torch.empty((2, nb, BLOCK, 2), dtype=torch.float32, device="cuda")
            chan.process_device([cap.data_ptr() for cap in caps], d_iq.data_ptr(), nb)
            chan.synchronize()
            iq[:, b0:b0 + nb] = d_iq.cpu().numpy()
    ps = [rx.make_params(mode=rx.DEMOD_USB, f_lo_cut=-100, f_hi_cut=100, agc_mode=0, psk31_enable=1, nco_freq=p[2])
          for p in placed]
    out = chain(ps, iq, want_psk=True)
    for s in range(2):
        chars = bytes(out["psk_chars"][s][out["psk_chars"][s] > 0])
        print("receiver %d decoded %r" % (s, chars))
        assert text.encode() in chars, (s, chars)


@pytest.mark.gpu
@pytest.mark.parametrize("kind, M", [("float", 64), ("q15", 320), ("real", 128)])
def test_argument_checks_on_a_device(kind, M):
    """EINVAL: a null or misaligned capture pointer, set_weights out of range or non-finite, set_weights on a
    single-input channelizer, each single-input process call on a diversity channelizer and the diversity call on a
    single-input one, each naming the entry point the channelizer takes"""
    import torch
    L = rx.lib()
    per_block = BLOCK * M // 2
    shape = (per_block,) if kind == "real" else (per_block, 2)
    dtype = torch.float32 if kind == "float" else torch.int16
    caps = [torch.zeros((per_block * 2 + 64,) + shape[1:], dtype=dtype, device="cuda") for _ in range(2)]
    iq = torch.zeros((2, 1, BLOCK, 2), dtype=torch.float32, device="cuda")
    misalign = 4 if kind == "float" else 8
    with rx.Channelizer(M, 2, n_inputs=2, **_opts(kind)) as ch:
        ch.set_map([0, 1])
        good = [c.data_ptr() for c in caps]
        ch.process_device(good, iq.data_ptr(), 1)
        ch.synchronize()
        for bad in ([good[0], None], [None, good[1]], [good[0], good[1] + misalign], [good[0] + misalign, good[1]]):
            arr = (C.c_void_p * 2)(*bad)
            assert L.t41rx_chan_process_device_diversity(ch._h, arr, C.c_void_p(iq.data_ptr()), 1, None) == EINVAL
        with pytest.raises(ValueError):
            ch.process_device(good[0], iq.data_ptr(), 1)
        with pytest.raises(rx.T41RxError, match="bad range"):
            ch.set_weights(np.ones((3, 2)))
        with pytest.raises(rx.T41RxError, match="bad range"):
            ch.set_weights(np.ones((1, 2)), first=2)
        for v in (np.nan, np.inf):
            with pytest.raises(rx.T41RxError, match="finite"):
                ch.set_weights(np.array([[1.0, v]]))
        for fn in ("t41rx_chan_process_device", "t41rx_chan_process_device_real", "t41rx_chan_process_device_q15"):
            assert getattr(L, fn)(ch._h, C.c_void_p(good[0]), C.c_void_p(iq.data_ptr()), 1, None) == EINVAL
            msg = L.t41rx_last_error()
            assert b"diversity channelizer takes t41rx_chan_process_device_diversity" in msg, (fn, msg)
    takes = {"float": b"t41rx_chan_process_device", "q15": b"t41rx_chan_process_device_q15",
             "real": b"t41rx_chan_process_device_real"}[kind]
    with rx.Channelizer(M, 2, **_opts(kind)) as single:
        arr = (C.c_void_p * 2)(*[c.data_ptr() for c in caps])
        assert L.t41rx_chan_process_device_diversity(single._h, arr, C.c_void_p(iq.data_ptr()), 1, None) == EINVAL
        assert b"channelizer takes " + takes in L.t41rx_last_error()
        w = (C.c_float * 4)(1, 0, 0, 0)
        assert L.t41rx_chan_set_weights(single._h, 0, 1, w) == EINVAL
        assert b"single-input" in L.t41rx_last_error()
