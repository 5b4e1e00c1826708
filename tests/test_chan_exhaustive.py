"""Channelizer parity on every output: all channels of all twelve kernel instances (complex float and int16 pairs at
M = 64 / 320 / 512 / 640, real int16 at M = 128 / 800 / 1024 / 1280), every row of a CTA's 16-output tile, the
fine-tuning phase past its wrap at 192000 outputs, the timing tool's bank shape, and INTEGRATION's device-resident step
loop.  The other channelizer modules check a handful of channels against the float64 formula with one pooled bound; a
bin swapped by the mixed-radix output positions, or an error confined to one tile row, passes them.

CPU tier: the all-channel float64 reference (chan_driver.reference_all_channels: polyphase sums, one M-point DFT per
output time, the (-1)^(k m) sign) against the direct formula (mix, convolution, decimation) at every M of every kind.

GPU tier: the kernels against that reference per receiver, with a bound B per instance (BOUND) set at about 3x the
worst per-channel error measured on an NVIDIA B200 (power limit 1000 W) and never above 1e-7 of the capture's RMS.
Measured worst per-channel error RMS / capture RMS (every channel, unshifted and shifted, the worst of two captures):
    float  64: 4.1e-8   320: 3.3e-8   512: 3.3e-8   640: 3.9e-8
    q15    64: 4.0e-8   320: 3.3e-8   512: 3.4e-8   640: 3.9e-8
    real  128: 3.2e-8   800: 2.6e-8  1024: 3.2e-8  1280: 3.6e-8
always on a channel that carries a tone (noise-only channels 0.6e-8 to 2.0e-8); tile rows' max / median 1.002 to 1.014;
across the wrap at most 3.7e-8 (float, q15 64) and 3.4e-8 (real 128); at the bank shape at most 0.8e-8.
"""
import ctypes as C

import numpy as np
import pytest

from chan_driver import channelize, cplx, reference_all_channels, reference_channel
from t41_sdr_b200 import rx, synth

BLOCK = rx.BLOCK
OUT_RATE = 192000
FILL = 12345.0
TILE = 16                     # output times per CTA (kChanTile): row mm = m mod 16 of a tile
K_TAPS = rx.CHAN_TAPS_PER_BRANCH
COMPLEX = (64, 320, 512, 640)
REAL = (128, 800, 1024, 1280)
KINDS = [("float", m) for m in COMPLEX] + [("q15", m) for m in COMPLEX] + [("real", m) for m in REAL]
# per-receiver bound on error RMS / capture RMS: about 3x the worst measured (module docstring), at most 1e-7
BOUND = {km: 1e-7 for km in KINDS}
BOUND.update({("real", 128): 9.5e-8, ("real", 800): 8e-8})
ROW_SPREAD = 1.5              # max / median of the 16 tile rows' error RMS (an FP32 emulation gives 1.00 to 1.02)


def _opts(kind):
    return {"real": kind == "real", "q15": kind == "q15"}


def _n_channels(kind, M):
    return M // 2 + 1 if kind == "real" else M


def _centre(kind, M, k):
    return rx.chan_centre_real(k) if kind == "real" else rx.chan_centre(M, k)


def _synth(kind, seed, M, n_blocks, signals, sigma, start_block=0):
    gen = {"float": synth.wideband, "q15": synth.wideband_q15, "real": synth.wideband_real}[kind]
    return gen(seed, M, n_blocks, signals, sigma=sigma, start_block=start_block)


def _capture(kind, M, n_blocks, seed, start_block=0):
    """six seeded tones, one near the top channel's centre, noise; for q15, full-scale samples (-32768 and 32767, in I
    and in Q) scattered through it.  Block b is the same whichever start_block / n_blocks it is generated in."""
    r = np.random.default_rng(seed)
    fs = synth.wideband_rate(M)
    lo = 0.0 if kind == "real" else -fs / 2
    sig = [("tone", float(r.uniform(lo, fs / 2)), {"amp": float(r.uniform(0.03, 0.15))}) for _ in range(6)]
    top = rx.chan_centre_real(M // 2) - 20000.0 if kind == "real" else rx.chan_centre(M, M // 2) + 1234.5
    sig.append(("tone", top, {"amp": 0.1}))
    blocks = []
    for b in range(start_block, start_block + n_blocks):
        s = _synth(kind, seed, M, 1, sig, 0.05, start_block=b)
        if kind == "q15":
            rb = np.random.default_rng([seed, b])
            for value in (-32768, 32767):
                idx = rb.choice(s.shape[0], 64, replace=False)
                s[idx, rb.integers(0, 2, idx.size)] = value
                s[rb.choice(s.shape[0], 8, replace=False)] = value
        blocks.append(s)
    return np.concatenate(blocks)


def _x(kind, capture):
    """the capture as the channelizer reads it, complex128"""
    if kind == "real":
        return capture.astype(np.float64) / 32768.0
    return cplx(capture) / (32768.0 if kind == "q15" else 1.0)


def _rms(x):
    return float(np.sqrt(np.mean(np.abs(x) ** 2)))


def _as_complex(iq):
    """iq [..., n_blocks, 2048, 2] float32 -> complex128 [..., n_blocks * 2048]"""
    z = iq[..., 0].astype(np.float64) + 1j * iq[..., 1].astype(np.float64)
    return z.reshape(z.shape[:-2] + (-1,))


def _rotor(shift, m):
    """exp(2 pi j (shift m mod 192000) / 192000) for receivers' shifts [R] and outputs m [n] (counted from creation)"""
    phi = (np.asarray(shift, np.int64)[:, None] * np.asarray(m, np.int64)[None, :]) % OUT_RATE
    return np.exp(2j * np.pi * phi / OUT_RATE)


def _bits_equal(a, b):
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


# ---------------------------------------------------------------- CPU tier

@pytest.mark.parametrize("kind, M", [("complex", m) for m in COMPLEX] + [("real", m) for m in REAL])
def test_all_channel_reference_matches_the_defining_formula(kind, M):
    """reference_all_channels against reference_channel (direct mix, convolution, decimation) on a seeded capture, at
    channels 0, 1, M/5, M/4, M/2, M - 1 (real: the rows 0 .. M/2 a real channelizer has): max |difference| <= 1e-12 of
    the channel's RMS over all outputs, and over the first 2K outputs alone, where the sums reach x[n < 0] = 0."""
    n_out = 96
    r = np.random.default_rng(3 + M)
    n = n_out * M // 2
    x = r.standard_normal(n) + (0.0 if kind == "real" else 1j * r.standard_normal(n))
    taps = rx.chan_taps(M)
    z_all = reference_all_channels(x, taps, M, n_out)
    assert z_all.shape == (M, n_out) and z_all.dtype == np.complex128
    for k in (0, 1, M // 5, M // 4, M // 2, M - 1):
        if kind == "real" and k > M // 2:
            continue
        want = reference_channel(x, taps, M, k, n_out)
        scale = _rms(want)
        err = np.abs(z_all[k] - want)
        assert err.max() <= 1e-12 * scale, (k, err.max() / scale)
        assert err[:2 * K_TAPS].max() <= 1e-12 * scale, (k, err[:2 * K_TAPS].max() / scale)


def test_all_channel_reference_of_a_real_capture_is_hermitian():
    """for real x the rows above M/2 mirror those below (z_{M-k} = conj z_k): the rows a real channelizer drops carry
    nothing new"""
    M, n_out = 128, 64
    x = np.random.default_rng(5).standard_normal(n_out * M // 2)
    z = reference_all_channels(x, rx.chan_taps(M), M, n_out)
    k = np.arange(1, M // 2)
    assert np.max(np.abs(z[M - k] - np.conj(z[k]))) <= 1e-12 * _rms(z)


# ---------------------------------------------------------------- GPU tier

def _every_channel_case(kind, M, seed):
    """receivers 0 .. n_ch-1 on channels 0 .. n_ch-1 unshifted, n_ch .. 2 n_ch-1 on the same channels with seeded
    shifts in (-192000, 192000) (+-1, +-96000 and +-191999 among them), one unmapped receiver last"""
    n_ch = _n_channels(kind, M)
    r = np.random.default_rng(seed)
    shifts = r.integers(-OUT_RATE + 1, OUT_RATE, n_ch)
    special = [1, -1, 96000, -96000, 191999, -191999]
    shifts[r.choice(n_ch, len(special), replace=False)] = special
    chmap = list(range(n_ch)) * 2 + [-1]
    return chmap, [0] * n_ch + [int(s) for s in shifts] + [777]


@pytest.mark.gpu
@pytest.mark.parametrize("kind, M", KINDS)
def test_every_channel_and_tile_row_against_float64(kind, M):
    """Every channel twice (unshifted, and with a seeded shift) and an unmapped receiver, 3 blocks in calls of 1 + 2, on
    a capture of tones and noise and on a noise-only one: per receiver, error RMS / capture RMS <= BOUND; on the noise
    capture, the error RMS of each tile row m mod 16 (rows 0 .. 7 are formed before the span's shared memory dies and
    8 .. 15 after it, real 12 and 4; odd rows carry the half-turn) within ROW_SPREAD of the rows' median.  The unshifted
    receivers are bit-identical to a channelizer in which no receiver is rotated (the kernel without fine tuning)."""
    T, calls = 3, [1, 2]
    n_ch = _n_channels(kind, M)
    chmap, shifts = _every_channel_case(kind, M, 600 + M + len(kind))
    n_recv = len(chmap)
    taps, m = rx.chan_taps(M), np.arange(T * BLOCK)
    noise = _synth(kind, 70 + M, M, T, [], 0.05)
    worst = []
    for name, capture in (("tones", _capture(kind, M, T, 500 + M)), ("noise", noise)):
        got = channelize(M, n_recv, capture, calls, [chmap, None], [shifts, None], fill=FILL, **_opts(kind))
        plain = channelize(M, n_ch, capture, calls, [list(range(n_ch)), None], fill=FILL, **_opts(kind))
        assert np.all(got[-1] == FILL)
        assert _bits_equal(got[:n_ch], plain)
        x = _x(kind, capture)
        z = reference_all_channels(x, taps, M, T * BLOCK)[:n_ch]
        want = np.concatenate([z, z * _rotor(shifts[n_ch:-1], m)])
        err = _as_complex(got[:-1]) - want
        ratio = np.sqrt(np.mean(np.abs(err) ** 2, axis=1)) / _rms(x)
        r_worst = int(np.argmax(ratio))
        print("%s M=%d %s: worst per-channel error RMS / capture RMS %.3g (channel %d, shift %d), median %.3g" % (
            kind, M, name, ratio[r_worst], chmap[r_worst], shifts[r_worst], np.median(ratio)))
        worst.append(ratio[r_worst])
        assert ratio.max() <= BOUND[(kind, M)], (name, chmap[r_worst], shifts[r_worst], ratio[r_worst])
        if name == "noise":
            rows = np.sqrt(np.mean(np.abs(err.reshape(err.shape[0], -1, TILE)) ** 2, axis=(0, 1)))
            spread = rows.max() / np.median(rows)
            print("%s M=%d noise: tile rows' error RMS max / median %.3f (row %d)" % (kind, M, spread, np.argmax(rows)))
            assert spread <= ROW_SPREAD, rows / np.median(rows)
    print("%s M=%d: worst per-channel ratio %.3g (bound %.3g)" % (kind, M, max(worst), BOUND[(kind, M)]))


WRAP_KINDS = [("float", 64), ("q15", 64), ("real", 128)]


@pytest.mark.gpu
@pytest.mark.parametrize("kind, M", WRAP_KINDS)
def test_fine_tuning_across_the_phase_wrap(kind, M):
    """200 blocks (409600 outputs: the phase counter, kept mod 192000, wraps at blocks 93.75 and 187.5) in calls of 37,
    37, 37, 1, 37, 37, 14 blocks, so that both wraps fall inside a call; shifts 1, -1, 12345, 191999, -96000 and 0 on
    channels that carry tones, and new shifts for three receivers after the first wrap.  Against the float64 formula
    rotated by a phase derived from the shift history alone: phi(m) = s0 m before the change at output mc, s0 mc +
    s1 (m - mc) after it (mod 192000, m counted from creation); per receiver error RMS / capture RMS <= BOUND.  Each
    call's capture is generated on its own (start_block), and so is the reference."""
    import torch
    calls = [37, 37, 37, 1, 37, 37, 14]
    change_before = 3                               # set_shift again before the 4th call (after block 111)
    T = sum(calls)
    per_block = BLOCK * M // 2
    last = M // 2 if kind == "real" else M - 1
    chans = [3, 3, M // 5, last, M // 2 - 1, M // 5]
    shift0 = [1, -1, 12345, 191999, -96000, 0]
    shift1 = [-191999, -1, 12345, 191999, 4321, 5000]
    sig = [("tone", _centre(kind, M, k) + 1000.0 * (i + 1), {"amp": 0.1}) for i, k in enumerate(sorted(set(chans)))]
    seed = 80 + M

    def blocks(b0, nb):
        return np.concatenate([_synth(kind, seed, M, 1, sig, 0.05, start_block=b) for b in range(b0, b0 + nb)])

    taps = rx.chan_taps(M)
    n_recv = len(chans)
    got = np.empty((n_recv, T, BLOCK, 2), np.float32)
    want = np.empty((n_recv, T * BLOCK), np.complex128)
    sum_x2, n_x = 0.0, 0
    mc = sum(calls[:change_before]) * BLOCK
    with rx.Channelizer(M, n_recv, **_opts(kind)) as ch:
        ch.set_map(chans)
        ch.set_shift(shift0)
        b0 = 0
        for i, nb in enumerate(calls):
            if i == change_before:
                ch.set_shift(shift1)
            lead = 1 if b0 > 0 else 0               # one block before the call: the reference's filter history
            cap = blocks(b0 - lead, nb + lead)
            d_cap = torch.from_numpy(np.ascontiguousarray(cap[lead * per_block:])).cuda()
            d_iq = torch.full((n_recv, nb, BLOCK, 2), FILL, dtype=torch.float32, device="cuda")
            ch.process_device(d_cap.data_ptr(), d_iq.data_ptr(), nb)
            ch.synchronize()
            got[:, b0:b0 + nb] = d_iq.cpu().numpy()
            x = _x(kind, cap)
            z = reference_all_channels(x, taps, M, (nb + lead) * BLOCK)[chans, lead * BLOCK:]
            m = np.arange(b0 * BLOCK, (b0 + nb) * BLOCK, dtype=np.int64)
            s0 = np.array(shift0, np.int64)[:, None]
            s1 = np.array(shift1, np.int64)[:, None]
            phi = np.where(m[None, :] < mc, s0 * m[None, :], s0 * mc + s1 * (m[None, :] - mc)) % OUT_RATE
            want[:, b0 * BLOCK:(b0 + nb) * BLOCK] = z * np.exp(2j * np.pi * phi / OUT_RATE)
            x_call = x[lead * per_block:]
            sum_x2 += float(np.sum(np.abs(x_call) ** 2))
            n_x += x_call.size
            b0 += nb
    ratio = np.sqrt(np.mean(np.abs(_as_complex(got) - want) ** 2, axis=1)) / np.sqrt(sum_x2 / n_x)
    print("%s M=%d over 200 blocks: per-receiver error RMS / capture RMS %s" % (kind, M, " ".join("%.3g" % v for v in ratio)))
    assert ratio.max() <= BOUND[(kind, M)], ratio


BANK_KINDS = [("float", 512), ("float", 640), ("real", 1024), ("real", 1280)]


@pytest.mark.gpu
@pytest.mark.parametrize("kind, M", BANK_KINDS)
def test_bench_bank_shape(kind, M):
    """tools/chan_timing.py's shape: 1024 receivers, 2 per channel on channels 0 .. 511, 64 blocks per call, a plain call
    and then a call with every receiver shifted (the tool's seeded shifts).  Compared on the device: the two receivers
    of a channel are bit-identical in the plain call; the 32 receivers of 16 seeded channels are bit-identical in both
    calls to a 32-receiver channelizer given the same entries in another order (an entry's output does not depend on
    the other entries); those receivers' first 2 blocks of each call pass the float64 check (BOUND)."""
    import torch
    S, T = 1024, 64
    per_block = BLOCK * M // 2
    n_cap = T * per_block
    dev = torch.device("cuda")
    g = torch.Generator(device=dev).manual_seed(11 + M)
    if kind == "real":
        d_cap = torch.randint(-3277, 3278, (n_cap,), generator=g, device=dev, dtype=torch.int16)
    else:
        d_cap = (0.1 * torch.randn((n_cap, 2), generator=g, device=dev)).contiguous()
    chmap = [(r // 2) % 512 for r in range(S)]
    rs = np.random.Generator(np.random.PCG64(2025))
    shifts = rs.integers(1, 96001, S) * rs.choice([-1, 1], S)
    r = np.random.default_rng(M)
    chans = np.sort(r.choice(512, 16, replace=False))
    picked = r.permutation(np.concatenate([2 * chans, 2 * chans + 1]))     # big-bank receivers, in the small bank's order
    small_map = [chmap[i] for i in picked]
    head = d_cap[:2 * per_block].cpu().numpy()
    tail = d_cap[n_cap - K_TAPS * M:].cpu().numpy()
    taps = rx.chan_taps(M)
    iq = torch.full((S, T, BLOCK, 2), float("nan"), dtype=torch.float32, device=dev)
    small_iq = torch.full((len(picked), T, BLOCK, 2), float("nan"), dtype=torch.float32, device=dev)
    idx = torch.from_numpy(picked).to(dev)
    with rx.Channelizer(M, S, **_opts(kind)) as big, rx.Channelizer(M, len(picked), **_opts(kind)) as small:
        big.set_map(chmap)
        small.set_map(small_map)
        for call in ("plain", "shifted"):
            if call == "shifted":
                big.set_shift(shifts)
                small.set_shift(shifts[picked])
            big.process_device(d_cap.data_ptr(), iq.data_ptr(), T)
            small.process_device(d_cap.data_ptr(), small_iq.data_ptr(), T)
            big.synchronize()
            small.synchronize()
            assert not bool(torch.isnan(iq).any()), call
            if call == "plain":
                assert torch.equal(iq[0::2].view(torch.int32), iq[1::2].view(torch.int32))
            assert torch.equal(iq.index_select(0, idx).view(torch.int32), small_iq.view(torch.int32)), call
            # float64 on the first 2 blocks of the call; the shifted call follows the plain one (the channelizer's
            # tail), and its phase restarts there: phi = s (m - m_done) with continuous phase from 0
            x = _x(kind, np.concatenate([tail, head]) if call == "shifted" else head)
            lead = 2 * K_TAPS if call == "shifted" else 0
            z = reference_all_channels(x, taps, M, lead + 2 * BLOCK)[:, lead:]
            got = _as_complex(small_iq[:, :2].cpu().numpy())
            want = z[small_map]
            if call == "shifted":
                want = want * _rotor(shifts[picked], np.arange(2 * BLOCK))
            ratio = np.sqrt(np.mean(np.abs(got - want) ** 2, axis=1)) / _rms(_x(kind, head))
            print("%s M=%d bank, %s call: worst error RMS / capture RMS %.3g" % (kind, M, call, ratio.max()))
            assert ratio.max() <= BOUND[(kind, M)], (call, ratio.max())


STEP_KINDS = [("float", 512), ("q15", 640), ("real", 1280)]


def _debug_bits(d):
    """every field of a receiver's debug state as its bytes (floats compared bit for bit, padding left out)"""
    return [(name, C.string_at(C.addressof(d) + getattr(rx.Debug, name).offset, getattr(rx.Debug, name).size))
            for name, _ in rx.Debug._fields_]


@pytest.mark.gpu
@pytest.mark.parametrize("kind, M", STEP_KINDS)
def test_device_resident_step_loop(kind, M):
    """INTEGRATION's loop: 4 steps of Channelizer.process_device(..., stream=s) and Receiver.process_device(...,
    cuda_stream=s) on one torch stream, the capture buffer refilled on s from pinned host memory each step, no host
    synchronisation until the end; 8 receivers placed by chan_place / chan_place_real (USB, LSB, AM, NFM).  Bit-identical
    to the same steps with the host round trip (channelize, then Receiver.process step by step): iq, audio and every
    field of each receiver's debug state."""
    import torch
    n_steps, nb, S = 4, 4, 8
    T = n_steps * nb
    per_block = BLOCK * M // 2
    capture = _capture(kind, M, T, 300 + M)
    fs = synth.wideband_rate(M)
    r = np.random.default_rng(M)
    modes = [rx.DEMOD_USB, rx.DEMOD_LSB, rx.DEMOD_AM, rx.DEMOD_NFM] * 2
    chmap, shifts, params = [], [], []
    for mode in modes:
        if kind == "real":
            ch, sh, nco = rx.chan_place_real(M, mode, float(r.uniform(0, fs / 2)))
        else:
            ch, sh, nco = rx.chan_place(M, mode, float(r.uniform(-fs / 2, fs / 2)))
        chmap.append(ch)
        shifts.append(sh)
        params.append(rx.make_params(mode=mode, nco_freq=nco))
    host = torch.from_numpy(capture.reshape((n_steps, nb * per_block) + capture.shape[1:])).pin_memory()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        d_cap = torch.empty(host.shape[1:], dtype=host.dtype, device="cuda")
        d_iq = torch.empty((S, nb, BLOCK, 2), dtype=torch.float32, device="cuda")
        d_audio = torch.empty((S, nb, BLOCK), dtype=torch.float32, device="cuda")
        iq_all = torch.empty((S, T, BLOCK, 2), dtype=torch.float32, device="cuda")
        audio_all = torch.empty((S, T, BLOCK), dtype=torch.float32, device="cuda")
    with rx.Channelizer(M, S, **_opts(kind)) as chan, rx.Receiver(S) as eng:
        chan.set_map(chmap)
        chan.set_shift(shifts)
        eng.set_params_each(params)
        with torch.cuda.stream(s):
            for i in range(n_steps):
                d_cap.copy_(host[i], non_blocking=True)
                chan.process_device(d_cap.data_ptr(), d_iq.data_ptr(), nb, stream=s.cuda_stream)
                eng.process_device(d_iq.data_ptr(), d_audio.data_ptr(), nb, cuda_stream=s.cuda_stream)
                iq_all[:, i * nb:(i + 1) * nb].copy_(d_iq)
                audio_all[:, i * nb:(i + 1) * nb].copy_(d_audio)
        s.synchronize()
        chan.synchronize()
        eng.synchronize()
        got_iq, got_audio = iq_all.cpu().numpy(), audio_all.cpu().numpy()
        got_debug = [_debug_bits(eng.debug(j)) for j in range(S)]
    want_iq = channelize(M, S, capture, [nb] * n_steps, [chmap] + [None] * (n_steps - 1),
                         [shifts] + [None] * (n_steps - 1), **_opts(kind))
    want_audio = np.empty_like(got_audio)
    with rx.Receiver(S) as eng:
        eng.set_params_each(params)
        for i in range(n_steps):
            want_audio[:, i * nb:(i + 1) * nb] = eng.process(want_iq[:, i * nb:(i + 1) * nb], flags=0)["audio"]
        want_debug = [_debug_bits(eng.debug(j)) for j in range(S)]
    assert _bits_equal(got_iq, want_iq)
    assert not np.any(np.isnan(got_audio)) and np.any(got_audio != 0.0)
    assert _bits_equal(got_audio, want_audio)
    for j in range(S):
        assert got_debug[j] == want_debug[j], j
