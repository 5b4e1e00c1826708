"""Drive a channelizer (t41_sdr_b200.rx.Channelizer, CUDA) over a capture, and the float64 references its output is
checked against: the defining formula of one channel, the fine-tuning rotation, the prototype's response."""
import numpy as np
from scipy.signal import fftconvolve

from t41_sdr_b200 import rx, synth

BLOCK = rx.BLOCK
OUT_RATE = 192000


def channelize(M, n_recv, capture, calls, maps, shifts=None, fill=12345.0, **kind):
    """One channelizer (kind: real= or q15=, as rx.Channelizer takes them) over `capture` in calls of calls[i] blocks;
    maps[i] and shifts[i] (each None or a list for receivers 0 ...) are set before call i.  Returns host iq
    [n_recv, sum(calls), 2048, 2]; rows of unmapped receivers keep `fill`."""
    import torch
    shifts = shifts or [None] * len(calls)
    per_block = BLOCK * M // 2
    d_cap = torch.from_numpy(np.ascontiguousarray(capture)).cuda()
    outs = []
    with rx.Channelizer(M, n_recv, **kind) as ch:
        b0 = 0
        for nb, chmap, sh in zip(calls, maps, shifts):
            if chmap is not None:
                ch.set_map(chmap)
            if sh is not None:
                ch.set_shift(sh)
            d_iq = torch.full((n_recv, nb, BLOCK, 2), fill, dtype=torch.float32, device="cuda")
            ch.process_device(d_cap[b0 * per_block:(b0 + nb) * per_block].data_ptr(), d_iq.data_ptr(), nb)
            ch.synchronize()
            outs.append(d_iq.cpu().numpy())
            b0 += nb
    return np.concatenate(outs, axis=1)


def reference_channel(x, taps, M, k, n_out):
    """float64 z_k[m] = conj(sum_i h[i] x[mD - i] exp(-2 pi j k (mD - i) / M)), m < n_out: direct mix, convolution,
    decimation.  x: capture from n = 0 (x[n < 0] = 0)."""
    D = M // 2
    n = np.arange(x.size)
    y = x * np.exp(-2j * np.pi * ((k * n) % M) / M)
    return np.conj(fftconvolve(y, taps.astype(np.float64))[:x.size][0:n_out * D:D])


def reference_all_channels(x, taps, M, n_out):
    """float64 z_k[m] of every channel k < M at once, m < n_out (complex128 [M, n_out]; a real capture's channels are
    rows 0 .. M/2): the defining formula factored as u_p[m] = sum_q h[p + qM] x[mD - p - qM] (x[n < 0] = 0), one
    M-point DFT of conj(u[m]) per output time, and the sign (-1)^(k m)."""
    D, K = M // 2, taps.size // M
    h = taps.astype(np.float64).reshape(K, M)
    xp = np.concatenate([np.zeros(K * M, np.complex128), np.asarray(x, np.complex128)])
    win = np.lib.stride_tricks.sliding_window_view(xp, M)      # win[j, t] = xp[j + t]
    m = np.arange(n_out)
    u = np.zeros((n_out, M), np.complex128)
    for q in range(K):
        # x[mD - p - qM] for p = 0 .. M-1 is win[mD + (K - 1 - q) M + 1] read backwards
        u += h[q] * win[m * D + (K - 1 - q) * M + 1][:, ::-1]
    z = np.fft.fft(np.conj(u), axis=1)
    z[1::2, 1::2] *= -1.0
    return z.T


def rotate(z, phase0, shift, m0=0):
    """float64 z[m] exp(2 pi j phi / 192000), phi = (phase0 + shift (m0 + m)) mod 192000 in integers."""
    m = np.arange(z.size, dtype=np.int64) + m0
    phi = (phase0 + shift * m) % OUT_RATE
    return z * np.exp(2j * np.pi * phi / OUT_RATE)


def response_db(taps, M, n_fft=1 << 20):
    H = np.fft.fft(taps.astype(np.float64), n_fft)
    f = np.fft.fftfreq(n_fft, 1.0 / synth.wideband_rate(M))
    return f, 20.0 * np.log10(np.maximum(np.abs(H), 1e-300))


def cplx(capture):
    return capture[:, 0].astype(np.float64) + 1j * capture[:, 1].astype(np.float64)


def error_ratio(got, want_by_receiver, x):
    """RMS of got[r] - want over the receivers r of want_by_receiver, over the RMS of the capture x"""
    err2, n_vals = 0.0, 0
    for r, want in want_by_receiver.items():
        g = got[r].reshape(-1, 2)
        err2 += np.sum((g[:, 0] - want.real) ** 2 + (g[:, 1] - want.imag) ** 2)
        n_vals += want.size
    return np.sqrt(err2 / n_vals) / np.sqrt(np.mean(np.abs(x) ** 2))


def chain(params, iq, want_psk=False):
    """the receiver chain (flags = 0) on iq [n_receivers, n_blocks, 2048, 2], with each receiver's debug state"""
    with rx.Receiver(len(params)) as eng:
        eng.set_params_each(params)
        out = eng.process(iq, want_psk=want_psk, flags=0)
        out["debug"] = [eng.debug(s) for s in range(len(params))]
    return out
