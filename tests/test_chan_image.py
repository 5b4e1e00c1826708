"""Image correction in the complex channelizers (DESIGN §3.12): receiver r on channel k gets rot_r(m) y_k[m],
y_k = z_k + c_k conj(z_kbar), kbar = (M - k) mod M, with per-channel coefficients set by hand or tracked on the GPU.

CPU tier: argument checks without a channelizer, ENODEV without a device, synth.iq_imbalance against its definition,
the model c_k = -conj(nu) / mu in float64, and the tracking rule in float64 (a strong tone's image to <= -100 dBc in
at most 3 calls at I/Q skews 0, 0.05 and 0.2 samples; the weak tone on the mirror side moves only by its own image,
within 0.01 dB up to a skew of 0.05 samples).

GPU tier, at each of the 8 complex (kind, M): every channel against float64 with seeded coefficients, unshifted and
shifted; zero coefficients and call splits bit for bit; q15 against float on s / 32768; tracking statistics against
float64 and the update against the rule applied on the host.  Then image rejection on imbalanced captures at int16
M = 640 and float M = 512, a calibration carried to a fresh channelizer, EINVAL on the real and diversity kinds, and a
weak USB receiver on a strong carrier's image frequency through the chain.
"""
import ctypes as C

import numpy as np
import pytest

import cases
import oracle_py as O
from chan_driver import chain, channelize, cplx, reference_all_channels, reference_channel
from t41_sdr_b200 import rx, synth

BLOCK = rx.BLOCK
OUT_RATE = 192000
EINVAL, ENODEV = -1, -4
FILL = 12345.0
KINDS = [("float", m) for m in (64, 320, 512, 640)] + [("q15", m) for m in (64, 320, 512, 640)]
BOUND = 1e-7                # error RMS / (RMS(x) (1 + |c_k|)), per receiver
G, PHI = 1.03, 2.0          # the imbalance of the rejection tests: gain and phase (degrees) on Q


def _mirror(M):
    return (-np.arange(M)) % M


def _mu_nu(g, phase_deg):
    e = np.exp(1j * np.deg2rad(phase_deg))
    return (1 + g * e) / 2, (1 - g * np.conj(e)) / 2


def _model_coef(g, phase_deg):
    mu, nu = _mu_nu(g, phase_deg)
    return -np.conj(nu) / mu


def _correct(z, coef):
    """float64 y_k = z_k + c_k conj(z_kbar) for z [M, n] (every channel)"""
    return z + coef[:, None] * np.conj(z[_mirror(z.shape[0])])


def _x(kind, capture):
    return cplx(capture) / (32768.0 if kind == "q15" else 1.0)


def _rms(x):
    return float(np.sqrt(np.mean(np.abs(x) ** 2)))


def _as_complex(iq):
    z = iq[..., 0].astype(np.float64) + 1j * iq[..., 1].astype(np.float64)
    return z.reshape(z.shape[:-2] + (-1,))


def _bits_equal(a, b):
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


def _rotor(shift, m):
    phi = (np.asarray(shift, np.int64)[:, None] * np.asarray(m, np.int64)[None, :]) % OUT_RATE
    return np.exp(2j * np.pi * phi / OUT_RATE)


def _tone(z, f, m0=0):
    """complex amplitude of exp(2 pi j f m / 192000) in z (f on a bin of len(z))"""
    m = m0 + np.arange(z.shape[-1])
    return np.mean(z * np.exp(-2j * np.pi * f * m / OUT_RATE), axis=-1)


def _capture(kind, M, n_blocks, seed):
    """seeded tones over the band (some pairs with a tone on one side only) and noise"""
    r = np.random.default_rng(seed)
    fs = synth.wideband_rate(M)
    sig = [("tone", float(r.uniform(-fs / 2, fs / 2)), {"amp": float(r.uniform(0.03, 0.15))}) for _ in range(6)]
    gen = synth.wideband_q15 if kind == "q15" else synth.wideband
    return gen(seed, M, n_blocks, sig, sigma=0.01)


def _coefs(M, seed):
    """seeded c_k: a third 0, a third small (|c| <= 0.03), a third |c| = 0.5; channels 0 and M/2 nonzero"""
    r = np.random.default_rng(seed)
    ph = np.exp(2j * np.pi * r.uniform(0, 1, M))
    pick = r.integers(0, 3, M)
    c = np.where(pick == 0, 0.0, np.where(pick == 1, r.uniform(0.001, 0.03, M), 0.5)) * ph
    c[0], c[M // 2] = 0.5 * ph[0], 0.02 * ph[M // 2]
    return c


def _every_channel_case(M, seed):
    """receivers 0 .. M-1 on channels 0 .. M-1 unshifted, M .. 2M-1 on the same channels with seeded shifts (+-1,
    +-96000 and +-191999 among them), one unmapped receiver last"""
    r = np.random.default_rng(seed)
    shifts = r.integers(-OUT_RATE + 1, OUT_RATE, M)
    special = [1, -1, 96000, -96000, 191999, -191999]
    shifts[r.choice(M, len(special), replace=False)] = special
    return list(range(M)) * 2 + [-1], [0] * M + [int(s) for s in shifts] + [777]


def channelize_image(M, n_recv, capture, calls, steps, fill=FILL, **kind):
    """chan_driver.channelize() with image correction: steps[i] (a dict or None) is applied before call i, keys "map",
    "shift", "image" (complex [n_channels] for every channel, or (first, complex array)), "track" (None: unchanged,
    False: off, a number: on with that dominance in dB).  Returns host iq [n_recv, sum(calls), 2048, 2], and per call
    the table after it (get_image) and, with tracking on, image_stats."""
    import torch
    per_block = BLOCK * M // 2
    d_cap = torch.from_numpy(np.ascontiguousarray(capture)).cuda()
    outs, tables, stats = [], [], []
    with rx.Channelizer(M, n_recv, **kind) as ch:
        b0, tracking = 0, False
        for nb, st in zip(calls, steps):
            st = st or {}
            if st.get("map") is not None:
                ch.set_map(st["map"])
            if st.get("shift") is not None:
                ch.set_shift(st["shift"])
            if st.get("image") is not None:
                im = st["image"]
                first, coef = im if isinstance(im, tuple) else (0, im)
                ch.set_image(coef, first)
            if st.get("track") is not None:
                tracking = st["track"] is not False
                ch.track_image(tracking, st["track"] if tracking else 20.0)
            d_iq = torch.full((n_recv, nb, BLOCK, 2), fill, dtype=torch.float32, device="cuda")
            ch.process_device(d_cap[b0 * per_block:(b0 + nb) * per_block].data_ptr(), d_iq.data_ptr(), nb)
            ch.synchronize()
            outs.append(d_iq.cpu().numpy())
            tables.append(ch.get_image())
            stats.append(ch.image_stats() if tracking else None)
            b0 += nb
    return np.concatenate(outs, axis=1), tables, stats


def _track_rule(coef, stats, dominance_db):
    """the update of DESIGN §3.12 on the host: float64 from the float32 table and the returned stats, rounded to
    float32 as the device rounds it"""
    M = coef.size
    T = 10.0 ** (dominance_db / 10.0)
    c = coef.astype(np.complex64).copy()
    for k in range(1, M // 2):
        ar, ai, pk, pb = stats[k]
        j, p = None, None
        if pk > 0 and pk >= T * pb:
            j, p = M - k, pk
        elif pb > 0 and pb >= T * pk:
            j, p = k, pb
        if j is not None:
            re = np.float32(np.float64(np.float32(c[j].real)) - ar / p)
            im = np.float32(np.float64(np.float32(c[j].imag)) - ai / p)
            c[j] = np.complex64(complex(re, im))
    return c


# ---------------------------------------------------------------- CPU tier

def test_image_entry_points_reject_a_null_channelizer():
    L = rx.lib()
    coef = (C.c_float * 4)(0, 0, 0, 0)
    stats = (C.c_double * 4)()
    assert L.t41rx_chan_set_image(None, 0, 1, coef) == EINVAL
    assert L.t41rx_chan_get_image(None, coef) == EINVAL
    assert L.t41rx_chan_track_image(None, 1, 20.0) == EINVAL
    assert L.t41rx_chan_image_stats(None, stats) == EINVAL
    assert b"null channelizer" in L.t41rx_last_error()


@pytest.mark.parametrize("q15", [False, True])
def test_image_channelizer_without_device_is_enodev(q15):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    h = C.c_void_p()
    create = rx.lib().t41rx_chan_create_q15 if q15 else rx.lib().t41rx_chan_create
    assert create(C.byref(h), 640, 4, 0) == ENODEV
    assert not h.value
    with pytest.raises(rx.T41RxError, match="no CUDA device"):
        rx.Channelizer(512, 4, q15=q15)


def test_iq_imbalance_against_its_definition():
    """I' = I, Q' = g (Q cos phi + I sin phi) delayed by the skew: checked on a sum of tones periodic in the capture
    (so the circular delay is the exact one) against the closed form, at skew 0 exactly, and the q15 form's rounding"""
    n = 4096
    t = np.arange(n)
    r = np.random.default_rng(3)
    bins = r.integers(-n // 2 + 1, n // 2, 6)
    amp = r.uniform(0.01, 0.2, 6) * np.exp(2j * np.pi * r.uniform(0, 1, 6))

    def s_at(tt):
        return sum(a * np.exp(2j * np.pi * b * tt / n) for a, b in zip(amp, bins))

    g, ph, d = 0.97, -3.5, 0.3
    phi = np.deg2rad(ph)
    for skew in (0.0, d):
        x = synth.iq_imbalance(s_at(t), g, ph, skew)
        sd = s_at(t - skew)
        want = s_at(t).real + 1j * g * (sd.imag * np.cos(phi) + sd.real * np.sin(phi))
        assert np.max(np.abs(x - want)) <= 1e-12
    s = s_at(t)
    x0 = synth.iq_imbalance(s, g, ph)
    assert np.array_equal(x0.real, s.real)
    mu, nu = _mu_nu(g, ph)
    assert np.max(np.abs(x0 - (mu * s + nu * np.conj(s)))) <= 1e-15
    q = synth.iq_imbalance_q15(s, g, ph, d)
    xd = synth.iq_imbalance(s, g, ph, d)
    assert np.array_equal(q[:, 0], np.clip(np.round(32768.0 * xd.real), -32768, 32767).astype(np.int16))
    assert np.array_equal(q[:, 1], np.clip(np.round(32768.0 * xd.imag), -32768, 32767).astype(np.int16))


def test_model_coefficient_removes_a_frequency_independent_image_in_float64():
    """x = mu s + nu conj(s): with c_k = -conj(nu) / mu on every channel, y_k = (conj(mu) + c nu) z_k(s) to the
    float64 floor (<= 1e-12 of the channel RMS); at g = 1.03, phi = 2 degrees, c = 0.01478 + 0.01745j"""
    c = _model_coef(G, PHI)
    assert abs(c - (0.01482 + 0.01745j)) <= 1e-4
    M, n_out = 64, 256
    r = np.random.default_rng(11)
    s = r.standard_normal(n_out * M // 2) + 1j * r.standard_normal(n_out * M // 2)
    x = synth.iq_imbalance(s, G, PHI)
    taps = rx.chan_taps(M)
    zs, zx = reference_all_channels(s, taps, M, n_out), reference_all_channels(x, taps, M, n_out)
    mu, nu = _mu_nu(G, PHI)
    y = _correct(zx, np.full(M, c))
    assert np.max(np.abs(y - (np.conj(mu) + c * nu) * zs)) <= 1e-12 * _rms(zs)
    # uncorrected, the image is there: conj(nu) conj(z_kbar(s)) in every channel
    assert np.max(np.abs(zx - np.conj(mu) * zs - np.conj(nu) * np.conj(zs[_mirror(M)]))) <= 1e-12 * _rms(zs)


def _track_float64(M, skew, n_calls, per_call=8, dominance_db=20.0):
    """float64 model of tracking on one imbalanced capture: a strong tone 1500 Hz into channel 5, a weak one (-60 dB)
    3000 Hz into its mirror channel (both on bins of a call); per call the image of the strong tone in dBc and the weak
    tone's level in y over its level in the uncorrected z (dB), and the most the correction can move it by returning
    the weak tone's own image from channel k (20 log10(1 + |c_kbar| |its image| / |it|), dB)"""
    k, n = 5, per_call * BLOCK
    kb = M - k
    sig = [("tone", rx.chan_centre(M, k) + 1500.0, {"amp": 0.5}),
           ("tone", rx.chan_centre(M, kb) + 3000.0, {"amp": 0.0005})]
    s = synth.wideband_sum(1, M, n_calls * per_call, sig)
    z = reference_all_channels(synth.iq_imbalance(s, G, PHI, skew), rx.chan_taps(M), M, n_calls * n)
    c = np.zeros(M, np.complex128)
    T = 10.0 ** (dominance_db / 10.0)
    out = []
    for call in range(n_calls):
        zz = z[:, call * n:(call + 1) * n]
        y = _correct(zz, c)
        car, img = abs(_tone(y[k], -1500.0)), abs(_tone(y[kb], 1500.0))
        weak = abs(_tone(y[kb], -3000.0)) / abs(_tone(zz[kb], -3000.0))
        self_image = abs(_tone(zz[k], 3000.0)) / abs(_tone(zz[kb], -3000.0))
        out.append((20 * np.log10(img / car), 20 * np.log10(weak), 20 * np.log10(1 + abs(c[kb]) * self_image)))
        for p in range(1, M // 2):
            A, Pk, Pb = np.sum(y[p] * y[M - p]), np.sum(np.abs(y[p]) ** 2), np.sum(np.abs(y[M - p]) ** 2)
            if Pk >= T * Pb:
                c[M - p] -= A / Pk
            elif Pb >= T * Pk:
                c[p] -= A / Pb
    return out


@pytest.mark.parametrize("skew", [0.0, 0.05, 0.2])
def test_tracking_rule_in_float64(skew):
    """the dominant-side rule, 16384-output calls at M = 64: the strong tone's image (about -30 dBc uncorrected) is
    <= -100 dBc after at most 3 calls, with I/Q skew as well.  The weak tone on the mirror side moves only by its own
    image, which the correction returns from channel k: within that bound at every skew, and within 0.01 dB up to a
    skew of 0.05 samples (at 0.2 samples it moves 0.016 dB, its bound being 0.021 dB)"""
    res = _track_float64(64, skew, 4)
    print("skew %.2f: " % skew + ", ".join("%.1f dBc (weak %+.5f dB, bound %.5f dB)" % r for r in res))
    assert res[0][0] > -40.0
    assert min(r[0] for r in res[1:4]) <= -100.0
    assert all(r[0] <= -100.0 for r in res[3:])
    assert all(abs(r[1]) <= r[2] * 1.001 + 1e-9 for r in res)
    if skew <= 0.05:
        assert all(abs(r[1]) <= 0.01 for r in res)


# ---------------------------------------------------------------- GPU tier

@pytest.mark.gpu
@pytest.mark.parametrize("kind, M", KINDS)
def test_every_channel_against_float64(kind, M):
    """seeded c_k (0, small, |c| = 0.5) on every channel, receivers unshifted and shifted: per receiver error RMS /
    (RMS(x) (1 + |c_k|)) <= 1e-7 against rot * (z_k + c_k conj(z_kbar)) in float64; the unmapped receiver keeps its
    fill"""
    T, calls = 3, [1, 2]
    chmap, shifts = _every_channel_case(M, 300 + M + len(kind))
    cap = _capture(kind, M, T, 50 + M)
    coef = _coefs(M, 7 + M)
    got, _, _ = channelize_image(M, len(chmap), cap, calls, [{"map": chmap, "shift": shifts, "image": coef}, None],
                                 q15=kind == "q15")
    assert np.all(got[-1] == FILL)
    x = _x(kind, cap)
    y = _correct(reference_all_channels(x, rx.chan_taps(M), M, T * BLOCK), coef.astype(np.complex64).astype(np.complex128))
    k = np.array(chmap[:-1])
    rot = np.concatenate([np.ones((M, T * BLOCK)), _rotor(shifts[M:-1], np.arange(T * BLOCK))])
    err = _as_complex(got[:-1]) - rot * y[k]
    ratio = np.sqrt(np.mean(np.abs(err) ** 2, axis=1)) / (_rms(x) * (1 + np.abs(coef[k])))
    w = int(np.argmax(ratio))
    print("%s M=%d: worst error RMS / (RMS(x) (1 + |c|)) %.3g (channel %d, |c| %.3f, shift %d), median %.3g" % (
        kind, M, ratio[w], chmap[w], abs(coef[chmap[w]]), shifts[w], np.median(ratio)))
    assert ratio.max() <= BOUND


@pytest.mark.gpu
@pytest.mark.parametrize("kind, M", KINDS)
def test_zero_coefficients_and_call_splits_are_bit_exact(kind, M):
    """all-zero coefficients set after nonzero ones give the uncorrected channelizer's bits; channels left at 0 beside
    corrected ones (every other channel) give them too, shifted or not; with fixed coefficients 1 + 2 + 5 blocks give
    the bits of one 8-block call"""
    q15 = kind == "q15"
    chmap, shifts = _every_channel_case(M, 500 + M)
    n = len(chmap)
    cap = _capture(kind, M, 8, 70 + M)
    coef = _coefs(M, 9 + M)
    plain = channelize(M, n, cap[:3 * BLOCK * M // 2], [1, 2], [chmap, None], [shifts, None], fill=FILL, q15=q15)
    got, _, _ = channelize_image(M, n, cap[:3 * BLOCK * M // 2], [1, 2],
                                 [{"map": chmap, "shift": shifts, "image": coef}, {"image": np.zeros(M)}], q15=q15)
    assert _bits_equal(got[:, 1:], plain[:, 1:])
    assert not _bits_equal(got[:M, :1], plain[:M, :1])
    half = coef.copy()
    half[0::2] = 0.0
    half[1::2] = np.where(half[1::2] == 0, 0.3, half[1::2])
    got, _, _ = channelize_image(M, n, cap[:3 * BLOCK * M // 2], [1, 2], [{"map": chmap, "shift": shifts, "image": half},
                                                                          None], q15=q15)
    even = np.array([k % 2 == 0 for k in chmap[:-1]] + [True])
    assert _bits_equal(got[even], plain[even])
    assert not _bits_equal(got[~even], plain[~even])
    small = np.r_[0:8, M // 2 - 3:M // 2 + 3, M - 8:M]            # fewer receivers for the split check
    cm, sh = [int(v) for v in small] * 2, [0] * small.size + [int(s) for s in np.array(shifts[M:2 * M])[small]]
    one, _, _ = channelize_image(M, len(cm), cap, [8], [{"map": cm, "shift": sh, "image": coef}], q15=q15)
    split, _, _ = channelize_image(M, len(cm), cap, [1, 2, 5], [{"map": cm, "shift": sh, "image": coef}, None, None],
                                   q15=q15)
    assert _bits_equal(one, split)


@pytest.mark.gpu
@pytest.mark.parametrize("M", [64, 320, 512, 640])
def test_q15_equals_float_on_s_over_32768(M):
    """the q15 channelizer with coefficients and shifts gives the float channelizer's bits on s / 32768, fixed and
    tracking"""
    chmap, shifts = _every_channel_case(M, 800 + M)
    cap = _capture("q15", M, 3, 90 + M)
    capf = (cap.astype(np.float32) / np.float32(32768.0)).astype(np.float32)
    coef = _coefs(M, 13 + M)
    steps = [{"map": chmap, "shift": shifts, "image": coef}, {"track": 20.0}]
    a, ta, sa = channelize_image(M, len(chmap), cap, [1, 2], steps, q15=True)
    b, tb, sb = channelize_image(M, len(chmap), capf, [1, 2], steps)
    assert _bits_equal(a, b)
    assert np.array_equal(ta[-1], tb[-1]) and np.array_equal(sa[-1], sb[-1])


@pytest.mark.gpu
@pytest.mark.parametrize("kind, M", KINDS)
def test_tracking_stats_and_update(kind, M):
    """tracking on over calls of 1 + 2 + 1 blocks: each call's image_stats match the float64 sums over that call's y
    (with the coefficients the call used) within 1e-5 relative; the table after each call is the rule applied on the
    host to the returned stats and the table before, bit for bit; the same schedule run twice gives identical bits"""
    q15 = kind == "q15"
    calls = [1, 2, 1]
    chmap = [3, M - 3, 0, M // 2, 1]
    cap = _capture(kind, M, sum(calls), 110 + M)
    coef = _coefs(M, 17 + M) * 0.02
    steps = [{"map": chmap, "image": coef, "track": 20.0}, None, None]
    got, tables, stats = channelize_image(M, len(chmap), cap, calls, steps, q15=q15)
    again, tables2, _ = channelize_image(M, len(chmap), cap, calls, steps, q15=q15)
    assert _bits_equal(got, again) and all(np.array_equal(a, b) for a, b in zip(tables, tables2))
    z = reference_all_channels(_x(kind, cap), rx.chan_taps(M), M, sum(calls) * BLOCK)
    before, b0, n_updates = coef.astype(np.complex64), 0, 0
    for nb, after, st in zip(calls, tables, stats):
        y = _correct(z[:, b0 * BLOCK:(b0 + nb) * BLOCK], before.astype(np.complex128))
        p = np.arange(M // 2 + 1)
        A = np.sum(y[p] * y[_mirror(M)[p]], axis=1)
        Pk, Pb = np.sum(np.abs(y[p]) ** 2, axis=1), np.sum(np.abs(y[_mirror(M)[p]]) ** 2, axis=1)
        scale = np.sqrt(Pk * Pb)
        assert np.max(np.abs(st[:, 0] + 1j * st[:, 1] - A) / scale) <= 1e-5
        assert np.max(np.abs(st[:, 2] / Pk - 1)) <= 1e-5 and np.max(np.abs(st[:, 3] / Pb - 1)) <= 1e-5
        want = _track_rule(before, st, 20.0)
        assert np.array_equal(after.astype(np.complex64), want)
        assert after[0] == before[0] and after[M // 2] == before[M // 2]
        n_updates += int(np.sum(want != before))
        before, b0 = want, b0 + nb
    print("%s M=%d: %d coefficient updates over %d calls" % (kind, M, n_updates, len(calls)))
    assert n_updates > 0


def _rejection_case(kind, M, skew, n_calls=4, per_call=4):
    """an imbalanced capture (g = 1.03, phi = 2 degrees, the skew): a strong tone 1500 Hz into channel k = M / 5 and a
    weak one (-60 dB) 3000 Hz into its mirror; receivers on k and kbar, tracking on from the first call; per call the
    image of the strong tone (dBc) and the weak tone's level over the uncorrected float64 one (dB)"""
    k = M // 5
    kb = M - k
    sig = [("tone", rx.chan_centre(M, k) + 1500.0, {"amp": 0.5}),
           ("tone", rx.chan_centre(M, kb) + 3000.0, {"amp": 0.0005})]
    s = synth.wideband_sum(21, M, n_calls * per_call, sig, sigma=1e-4)
    if kind == "q15":
        cap = synth.iq_imbalance_q15(s, G, PHI, skew)
    else:
        x = synth.iq_imbalance(s, G, PHI, skew)
        cap = np.stack([x.real, x.imag], axis=-1).astype(np.float32)
    return k, kb, cap


def _levels(y, yb, zb):
    img = 20 * np.log10(abs(_tone(yb, 1500.0)) / abs(_tone(y, -1500.0)))
    return img, 20 * np.log10(abs(_tone(yb, -3000.0)) / abs(_tone(zb, -3000.0)))


def _self_image_bound(c_kb, z, zb):
    """the most a correction c_kb moves the weak tone by returning its own image from channel k (dB)"""
    return 20 * np.log10(1 + abs(c_kb) * abs(_tone(z, 3000.0)) / abs(_tone(zb, -3000.0)))


@pytest.mark.gpu
@pytest.mark.parametrize("kind, M", [("q15", 640), ("float", 512)])
@pytest.mark.parametrize("skew", [0.0, 0.1])
def test_image_rejection_on_an_imbalanced_capture(kind, M, skew):
    """tracking: the image is <= -90 dBc within 4 calls and the weak tone on the mirror side is unchanged within
    0.01 dB, or with skew within what its own image returned by the correction can move it (test_tracking_rule_in_
    float64; the skew's phase is larger here, at 0.2 of the capture rate); the model c_k = -conj(nu) / mu set by hand: the image within 1 dB of the float64 model's (or both below
    -110 dBc, where float32 rounding and the capture's noise decide)"""
    per_call, n_calls = 4, 4
    k, kb, cap = _rejection_case(kind, M, skew, n_calls, per_call)
    n = per_call * BLOCK
    tracked, tables, _ = channelize_image(M, 2, cap, [per_call] * n_calls, [{"map": [k, kb], "track": 20.0}] + [None] * 3,
                                          q15=kind == "q15")
    z = reference_all_channels(_x(kind, cap), rx.chan_taps(M), M, n_calls * n)
    res = [_levels(_as_complex(tracked[0, c * per_call:(c + 1) * per_call]),
                   _as_complex(tracked[1, c * per_call:(c + 1) * per_call]), z[kb, c * n:(c + 1) * n])
           for c in range(n_calls)]
    bound = [0.0] + [_self_image_bound(tables[c - 1][kb], z[k, c * n:(c + 1) * n], z[kb, c * n:(c + 1) * n])
                     for c in range(1, n_calls)]
    coef = np.full(M, _model_coef(G, PHI))
    fixed, _, _ = channelize_image(M, 2, cap[:2 * per_call * BLOCK * M // 2], [per_call, per_call],
                                   [{"map": [k, kb], "image": coef}, None], q15=kind == "q15")
    y = _correct(z[:, n:2 * n], coef.astype(np.complex64).astype(np.complex128))
    model = _levels(y[k], y[kb], z[kb, n:2 * n])[0]
    got = _levels(_as_complex(fixed[0, per_call:]), _as_complex(fixed[1, per_call:]), z[kb, n:2 * n])[0]
    print("%s M=%d skew %.1f: tracked %s; model c: %.1f dBc (float64 %.1f dBc)" % (
        kind, M, skew, ", ".join("%.1f dBc / weak %+.4f dB (bound %.4f)" % (r + (b,)) for r, b in zip(res, bound)),
        got, model))
    assert res[0][0] > -45.0
    assert min(r[0] for r in res) <= -90.0 and res[-1][0] <= -90.0
    assert all(abs(r[1]) <= max(0.01 if skew == 0.0 else 0.0, b + 1e-4) for r, b in zip(res, bound))
    assert abs(got - model) <= 1.0 or max(got, model) <= -110.0


@pytest.mark.gpu
@pytest.mark.parametrize("kind, M", [("q15", 640), ("float", 512)])
def test_calibration_carried_to_a_fresh_channelizer(kind, M):
    """get_image after tracking, set_image into a fresh channelizer given the tracked one's tail: the next call of
    both (tracking off) is bit-identical"""
    import torch
    per_call = 2
    k, kb, cap = _rejection_case(kind, M, 0.1, 3, per_call)
    per_block = BLOCK * M // 2
    d = torch.from_numpy(cap).cuda()
    q15 = kind == "q15"
    outs = []
    with rx.Channelizer(M, 2, q15=q15) as a:
        a.set_map([k, kb])
        a.track_image(True, 20.0)
        iq = torch.zeros((2, per_call, BLOCK, 2), dtype=torch.float32, device="cuda")
        for c in range(2):
            a.process_device(d[c * per_call * per_block:].data_ptr(), iq.data_ptr(), per_call)
        a.track_image(False)
        table = a.get_image()
        assert np.any(table != 0)
        a.process_device(d[2 * per_call * per_block:].data_ptr(), iq.data_ptr(), per_call)
        a.synchronize()
        outs.append(iq.cpu().numpy())
    with rx.Channelizer(M, 2, q15=q15) as b:
        b.set_map([k, kb])
        iq = torch.zeros((2, per_call, BLOCK, 2), dtype=torch.float32, device="cuda")
        # the same tail: run the first two calls' capture uncorrected, then the calibration
        for c in range(2):
            b.process_device(d[c * per_call * per_block:].data_ptr(), iq.data_ptr(), per_call)
        b.set_image(table)
        assert np.array_equal(b.get_image(), table)
        b.process_device(d[2 * per_call * per_block:].data_ptr(), iq.data_ptr(), per_call)
        b.synchronize()
        outs.append(iq.cpu().numpy())
    assert _bits_equal(outs[0], outs[1])


@pytest.mark.gpu
@pytest.mark.parametrize("kind, M", [("float", 64), ("q15", 320)])
def test_argument_checks_on_a_device(kind, M):
    """EINVAL: set_image out of range or non-finite, a dominance outside [3, 60] dB, image_stats before any tracking
    call; every image entry point on a real and on a diversity channelizer, saying why"""
    L = rx.lib()
    q15 = kind == "q15"
    with rx.Channelizer(M, 2, q15=q15) as ch:
        with pytest.raises(rx.T41RxError, match="bad range"):
            ch.set_image(np.zeros(M + 1))
        with pytest.raises(rx.T41RxError, match="bad range"):
            ch.set_image(np.zeros(2), first=M - 1)
        with pytest.raises(rx.T41RxError, match="bad range"):
            ch.set_image(np.zeros(1), first=-1)
        for v in (np.nan, np.inf, -np.inf):
            with pytest.raises(rx.T41RxError, match="finite"):
                ch.set_image([complex(v, 0)], first=3)
            with pytest.raises(rx.T41RxError, match="finite"):
                ch.set_image([complex(0, v)], first=3)
        for db in (2.9, 60.5, -20.0, float("nan")):
            with pytest.raises(rx.T41RxError, match="dominance_db"):
                ch.track_image(True, db)
        with pytest.raises(rx.T41RxError, match="no call has run with tracking on"):
            ch.image_stats()
        ch.track_image(False, float("nan"))        # the dominance is not read when turning tracking off
        ch.set_image([0.1 + 0.2j], first=M - 1)
        want = np.zeros(M, np.complex64)
        want[M - 1] = np.complex64(0.1 + 0.2j)
        assert np.array_equal(ch.get_image(), want)
    coef = (C.c_float * 2)(0.1, 0.0)
    stats = (C.c_double * (4 * (M + 1)))()
    others = [(rx.Channelizer(2 * M if M == 64 else 800, 2, real=True), b"a real channelizer has no image correction"),
              (rx.Channelizer(M, 2, q15=q15, n_inputs=2), b"a diversity channelizer has no image correction")]
    for ch, msg in others:
        with ch:
            for rc in (L.t41rx_chan_set_image(ch._h, 0, 1, coef), L.t41rx_chan_get_image(ch._h, coef),
                       L.t41rx_chan_track_image(ch._h, 1, 20.0), L.t41rx_chan_image_stats(ch._h, stats)):
                assert rc == EINVAL
                assert msg in L.t41rx_last_error()


def _debug_ints(d):
    return [getattr(d, f) for f in cases.DEBUG_INT_FIELDS]


@pytest.mark.gpu
def test_weak_usb_receiver_on_a_carriers_image_through_the_chain_q15_640():
    """sc16 at 61.44 MS/s (M = 640), g = 1.03, phi = 2 degrees: a carrier at F and a weak USB signal 60 dB below it
    whose receiver (chan_place, dial -F - 1000 Hz) hears the carrier's image as a 1000 Hz tone and the signal at
    1679.6875 Hz (both on bins of a call, as the tracking sums want).  Tracking settles over 2 calls of 8 blocks; the
    next 16 blocks (calls of 8, tracking on) go through the chain against the chain fed with the float64 channel of the
    balanced capture (the quantised capture with the imbalance undone, times the wanted's gain through imbalance and
    correction): audio SNR >= 90 dB after block 2 and the discrete state identical.  The image's audio tone with
    tracking off and on is reported.  What is left of the image comes from the capture's quantisation noise in each
    call's estimate of c_kbar, so longer calls leave less"""
    import torch
    M, settle, T, step = 640, 16, 16, 8
    F = rx.chan_centre(M, 100) + 23437.5
    dial = -F - 1000.0
    ch, shift, nco = rx.chan_place(M, rx.DEMOD_USB, dial)
    f_sig = 1679.6875
    sig = [("tone", F, {"amp": 0.9}), ("tone", dial + f_sig, {"amp": 0.0009})]
    s = synth.wideband_sum(41, M, settle + T, sig)      # the capture's noise is its quantisation
    cap = synth.iq_imbalance_q15(s, G, PHI)
    per_block = BLOCK * M // 2
    d = torch.from_numpy(cap).cuda()
    iqs = []
    for track in (False, True):
        out = np.empty((1, T, BLOCK, 2), np.float32)
        with rx.Channelizer(M, 1, q15=True) as chan:
            chan.set_map([ch])
            chan.set_shift([shift])
            if track:
                chan.track_image(True, 20.0)
            iq = torch.empty((1, step, BLOCK, 2), dtype=torch.float32, device="cuda")
            for b0 in range(0, settle + T, step):
                chan.process_device(d[b0 * per_block:].data_ptr(), iq.data_ptr(), step)
                chan.synchronize()
                if b0 >= settle:
                    out[:, b0 - settle:b0 - settle + step] = iq.cpu().numpy()
            if track:
                c_kb = chan.get_image()[ch]
        iqs.append(out)
    # the balanced capture: the quantised one with the imbalance undone in float64
    mu, nu = _mu_nu(G, PHI)
    xq = _x("q15", cap)
    bal = (np.conj(mu) * xq - nu * np.conj(xq)) / (abs(mu) ** 2 - abs(nu) ** 2)
    z = reference_channel(bal, rx.chan_taps(M), M, ch, (settle + T) * BLOCK)[settle * BLOCK:]
    ref = (np.conj(mu) + _model_coef(G, PHI) * nu) * z * _rotor([shift], settle * BLOCK + np.arange(T * BLOCK))[0]
    ref_iq = np.empty((1, T, BLOCK, 2), np.float32)
    ref_iq[0, ..., 0] = ref.real.reshape(T, BLOCK)
    ref_iq[0, ..., 1] = ref.imag.reshape(T, BLOCK)
    ps = [rx.make_params(mode=rx.DEMOD_USB, nco_freq=nco, agc_mode=0)]
    off, on, want = chain(ps, iqs[0]), chain(ps, iqs[1]), chain(ps, ref_iq)
    snr = O.snr_db(want["audio"][0, 2:], on["audio"][0, 2:])
    t = np.arange(want["audio"][0, 4:].size) / 192000.0
    win = np.hanning(t.size)

    def level(a, f):
        return abs(np.sum(win * a["audio"][0, 4:].reshape(-1) * np.exp(-2j * np.pi * f * t)))

    img_off = 20 * np.log10(level(off, 1000.0) / level(off, f_sig))
    img_on = 20 * np.log10(max(level(on, 1000.0), 1e-30) / level(on, f_sig))
    print("q15 640 through the chain: c_kbar %s (model %s); carrier image %.1f dB (off) / %.1f dB (on) relative to "
          "the weak signal; tracked receiver audio SNR %.1f dB" % (np.round(c_kb, 6), np.round(_model_coef(G, PHI), 6),
                                                                    img_off, img_on, snr))
    assert img_off > 0.0
    assert snr >= 90.0
    assert _debug_ints(on["debug"][0]) == _debug_ints(want["debug"][0])
