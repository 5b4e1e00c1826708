"""Channelizer timing on one GPU (DESIGN §3.7 - 3.9): M = 512 channels, 1024 receivers (2 per channel), 64 blocks per call.

    python tools/chan_timing.py [--calls 20] [--warmup 3] [--shift] [--real] [--q15] [--rates] [--diversity N] [--image]
                                [--json OUT]

Prints the card's name and power limit (a query), then CUDA-event times of
  - t41rx_chan_process_device alone (capture 268 MB, larger than the 126 MB L2; iq out 1 GiB),
  - the C2 chain step alone (t41rx_process_device on the channelizer's output, USB / AM mix, one row per step),
  - channelize + chain on one stream,
  - with --shift, t41rx_chan_process_device again after every receiver has been given its own fine-tuning shift
    (t41rx_chan_set_shift, seeded, 0 < |shift| <= 96 kHz as t41rx_chan_place gives them), in the same run,
  - with --real, t41rx_chan_process_device_real on a real int16 capture at M = 1024 (98.304 MS/s, the same 1024
    receivers on channels 0 ... 511, 64 blocks: 134 MB of capture, also larger than the L2), and with --shift also
    with every receiver shifted,
  - with --q15, at the same M and 1024 receivers: t41rx_chan_process_device_q15 on an interleaved int16 capture (134 MB
    at M = 512), and what a user of the float call does with such a capture: int16 -> float32 / 32768 with torch into
    a float capture, then t41rx_chan_process_device (with --shift also the q15 call with every receiver shifted),
  - with --rates (DESIGN §3.10), every channel count beside its power-of-two neighbour: the complex float call at
    M = 320, 512 and 640 and the real call at M = 800, 1024 and 1280, each without and with every receiver shifted.
    The same 1024 receivers, 2 per channel on channels 0 ... 511 (at M = 320 and 800, which have fewer channels, on
    channel (r / 2) mod 320 and mod 401), 64 blocks per call; the calls alternate between two captures, so that the
    captures a size reads (2 x 105 MB at real M = 800, more elsewhere) do not fit the L2,
  - with --diversity N (DESIGN §3.11), an N-input diversity call against the single-input call of the same kind and
    shape: complex float and int16 pairs at M = 512, real at M = 1024 and 1280; the same 1024 receivers, 2 per channel,
    64 blocks per call, every receiver shifted and given seeded weights on every input (none of them the default).  The
    single-input call alternates between two of the N captures; the N-input call reads all N (each at least 134 MB),
  - with --image (DESIGN §3.12), image correction against the plain call of the same channelizer: complex float at
    M = 512 and int16 pairs at M = 640; the same 1024 receivers, 2 per channel, 64 blocks per call, every receiver
    shifted; the plain call (every c_k 0), fixed seeded coefficients on every channel, tracking on (from those
    coefficients), and the plain call again, in that order on one channelizer,
each over --calls calls after --warmup calls.  Bytes moved are computed from shapes (capture read once, every mapped
receiver's iq written once) and given as a share of the B200's 7.7 TB/s HBM3e.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from t41_sdr_b200 import rx  # noqa: E402

HBM_BYTES_PER_S = 7.7e12


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown (nvidia-smi failed)"


def c2_params(n):
    r = np.random.Generator(np.random.PCG64(2024))
    out = []
    for k in range(n):
        nco = int(r.integers(-20000, 20001))
        if k % 2 == 0:
            out.append(rx.make_params(mode=rx.DEMOD_USB, f_lo_cut=300, f_hi_cut=3000, nco_freq=nco, agc_mode=1))
        else:
            out.append(rx.make_params(mode=rx.DEMOD_AM, nco_freq=nco, agc_mode=1))
    return out


def rate_table(g, dev, iq, sp, timed, shifts, S, T):
    """the --rates measurements: per (kind, M) the call's time without and with every receiver shifted, and each
    mixed-radix size against its power-of-two neighbour, per call and per capture sample"""
    import torch
    out = {}
    for kind, M in (("complex", 320), ("complex", 512), ("complex", 640), ("real", 800), ("real", 1024), ("real", 1280)):
        real = kind == "real"
        n_cap = T * rx.BLOCK * M // 2
        if real:
            caps = [torch.randint(-3277, 3278, (n_cap,), generator=g, device=dev, dtype=torch.int16) for _ in range(2)]
        else:
            caps = [(0.1 * torch.randn((n_cap, 2), generator=g, device=dev)).contiguous() for _ in range(2)]
        n_chan = M // 2 + 1 if real else M
        chan = rx.Channelizer(M, S, real=real)
        chan.set_map([(r // 2) % min(512, n_chan) for r in range(S)])
        calls = [0]

        def do():
            chan.process_device(caps[calls[0] % 2].data_ptr(), iq.data_ptr(), T, stream=sp)
            calls[0] += 1

        t = timed(do)
        chan.set_shift(shifts)
        t_shift = timed(do)
        chan.synchronize()
        chan.close()
        cap_bytes = n_cap * (2 if real else 8)
        moved = cap_bytes + S * T * rx.BLOCK * 8
        out["%s_%d" % (kind, M)] = {
            "capture_msps": M * 96e3 / 1e6, "capture_bytes": cap_bytes, "bytes_moved": moved,
            "chan_ms": {"median": t[0], "min": t[1], "max": t[2]},
            "all_shifted_ms": {"median": t_shift[0], "min": t_shift[1], "max": t_shift[2]},
            "ns_per_capture_sample": t[0] * 1e6 / n_cap,
            "all_shifted_ns_per_capture_sample": t_shift[0] * 1e6 / n_cap,
            "hbm_share_of_7p7_tbs": moved / (t[0] * 1e-3) / HBM_BYTES_PER_S}
        del caps
    for new, old in (("complex_320", "complex_512"), ("complex_640", "complex_512"), ("real_800", "real_1024"),
                     ("real_1280", "real_1024")):
        n, o = out[new], out[old]
        for key, ms in (("", "chan_ms"), ("all_shifted_", "all_shifted_ms")):
            n[key + "per_sample_over_" + old] = n[key + "ns_per_capture_sample"] / o[key + "ns_per_capture_sample"]
            n[key + "goal_per_sample_le_" + old] = n[key + "ns_per_capture_sample"] <= o[key + "ns_per_capture_sample"]
            if new in ("complex_640", "real_1280"):
                n[key + "call_over_" + old] = n[ms]["median"] / o[ms]["median"]
                n[key + "goal_call_le_1p25_of_" + old] = n[ms]["median"] <= 1.25 * o[ms]["median"]
    return out


def diversity_table(g, dev, iq, sp, timed, shifts, S, T, n_inputs):
    """the --diversity measurements: per (kind, M) the single-input call (before and after) and the n_inputs diversity
    call, in the same run, and their ratio against the goal (at most 2.5 x)"""
    import torch
    r = np.random.Generator(np.random.PCG64(2026))
    w = (0.2 + r.uniform(0, 1, (S, n_inputs))) * np.exp(2j * np.pi * r.uniform(0, 1, (S, n_inputs)))
    chmap = [(i // 2) % 512 for i in range(S)]
    out = {}
    for kind, M in (("complex", 512), ("q15", 512), ("real", 1024), ("real", 1280)):
        real, q15 = kind == "real", kind == "q15"
        n_cap = T * rx.BLOCK * M // 2
        if real:
            caps = [torch.randint(-3277, 3278, (n_cap,), generator=g, device=dev, dtype=torch.int16) for _ in range(n_inputs)]
        elif q15:
            caps = [torch.randint(-3277, 3278, (n_cap, 2), generator=g, device=dev, dtype=torch.int16) for _ in range(n_inputs)]
        else:
            caps = [(0.1 * torch.randn((n_cap, 2), generator=g, device=dev)).contiguous() for _ in range(n_inputs)]
        single = rx.Channelizer(M, S, real=real, q15=q15)
        div = rx.Channelizer(M, S, real=real, q15=q15, n_inputs=n_inputs)
        for c in (single, div):
            c.set_map(chmap)
            c.set_shift(shifts)
        div.set_weights(w)
        ptrs = [c.data_ptr() for c in caps]
        calls = [0]

        def do_single():
            single.process_device(ptrs[calls[0] % 2], iq.data_ptr(), T, stream=sp)
            calls[0] += 1

        def do_div():
            div.process_device(ptrs, iq.data_ptr(), T, stream=sp)

        t_single = timed(do_single)
        t_div = timed(do_div)
        t_single2 = timed(do_single)
        for c in (single, div):
            c.synchronize()
            c.close()
        cap_bytes = caps[0].numel() * caps[0].element_size()
        iq_bytes = S * T * rx.BLOCK * 8
        moved_single = cap_bytes + iq_bytes
        # every pass reads its capture; pass 0 writes iq, each later pass reads and writes it
        moved_div = n_inputs * cap_bytes + iq_bytes + (n_inputs - 1) * 2 * iq_bytes
        ratio = t_div[0] / min(t_single[0], t_single2[0])
        out["%s_%d" % (kind, M)] = {
            "capture_bytes_per_input": cap_bytes,
            "single_ms": {"median": t_single[0], "min": t_single[1], "max": t_single[2]},
            "single_again_ms": {"median": t_single2[0], "min": t_single2[1], "max": t_single2[2]},
            "diversity_ms": {"median": t_div[0], "min": t_div[1], "max": t_div[2]},
            "diversity_over_single": ratio,
            "goal_le_2p5_x_single": ratio <= 2.5,
            "single_bytes_moved": moved_single, "diversity_bytes_moved": moved_div,
            "single_hbm_share_of_7p7_tbs": moved_single / (t_single[0] * 1e-3) / HBM_BYTES_PER_S,
            "diversity_hbm_share_of_7p7_tbs": moved_div / (t_div[0] * 1e-3) / HBM_BYTES_PER_S}
        del caps
    return out


def image_table(g, dev, iq, sp, timed, shifts, S, T):
    """the --image measurements: per (kind, M) the plain call, fixed coefficients and tracking, and their ratios to
    the plain call against the goals (at most 1.10 x fixed, 1.25 x tracking)"""
    import torch
    r = np.random.Generator(np.random.PCG64(2027))
    chmap = [(i // 2) % 512 for i in range(S)]
    out = {}
    for kind, M in (("complex", 512), ("q15", 640)):
        q15 = kind == "q15"
        n_cap = T * rx.BLOCK * M // 2
        if q15:
            cap = torch.randint(-3277, 3278, (n_cap, 2), generator=g, device=dev, dtype=torch.int16)
        else:
            cap = (0.1 * torch.randn((n_cap, 2), generator=g, device=dev)).contiguous()
        chan = rx.Channelizer(M, S, q15=q15)
        chan.set_map(chmap)
        chan.set_shift(shifts)

        def do():
            chan.process_device(cap.data_ptr(), iq.data_ptr(), T, stream=sp)

        t_plain = timed(do)
        chan.set_image(0.03 * r.uniform(0.1, 1, M) * np.exp(2j * np.pi * r.uniform(0, 1, M)))
        t_fixed = timed(do)
        chan.track_image(True, 20.0)
        t_track = timed(do)
        chan.track_image(False)
        chan.set_image(np.zeros(M))
        t_plain2 = timed(do)
        chan.synchronize()
        chan.close()
        base = min(t_plain[0], t_plain2[0])
        out["%s_%d" % (kind, M)] = {
            "capture_bytes": cap.numel() * cap.element_size(),
            "plain_ms": {"median": t_plain[0], "min": t_plain[1], "max": t_plain[2]},
            "fixed_ms": {"median": t_fixed[0], "min": t_fixed[1], "max": t_fixed[2]},
            "tracking_ms": {"median": t_track[0], "min": t_track[1], "max": t_track[2]},
            "plain_again_ms": {"median": t_plain2[0], "min": t_plain2[1], "max": t_plain2[2]},
            "fixed_over_plain": t_fixed[0] / base, "goal_fixed_le_1p10": t_fixed[0] <= 1.10 * base,
            "tracking_over_plain": t_track[0] / base, "goal_tracking_le_1p25": t_track[0] <= 1.25 * base}
        del cap
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--channels", type=int, default=512)
    ap.add_argument("--receivers", type=int, default=1024)
    ap.add_argument("--blocks", type=int, default=64)
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--shift", action="store_true", help="also time the channelizer with every receiver shifted")
    ap.add_argument("--real", action="store_true", help="also time the real M = 1024 channelizer")
    ap.add_argument("--q15", action="store_true", help="also time the q15 channelizer and torch conversion + float")
    ap.add_argument("--rates", action="store_true", help="also time every channel count beside its power-of-two neighbour")
    ap.add_argument("--diversity", type=int, default=0, metavar="N",
                    help="also time an N-input diversity call against the single-input call (N = 2 ... 4)")
    ap.add_argument("--image", action="store_true", help="also time image correction, fixed and tracking")
    ap.add_argument("--json", default=None, help="also write the result here")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("chan_timing: no CUDA device")
    M, S, T = a.channels, a.receivers, a.blocks
    per_block = rx.BLOCK * M // 2
    n_cap = T * per_block
    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev).manual_seed(1)
    capture = (0.1 * torch.randn((n_cap, 2), generator=g, device=dev)).contiguous()
    iq = torch.empty((S, T, rx.BLOCK, 2), dtype=torch.float32, device=dev)
    audio = torch.empty((S, T, rx.BLOCK), dtype=torch.float32, device=dev)
    spec = torch.empty((S, 1, rx.SPECTRUM_RES), dtype=torch.int16, device=dev)
    wf = torch.empty((S, 1, rx.SPECTRUM_RES), dtype=torch.uint16, device=dev)
    stream = torch.cuda.Stream(device=dev)
    sp = stream.cuda_stream

    chan = rx.Channelizer(M, S)
    chan.set_map([(r // 2) % M for r in range(S)])
    eng = rx.Receiver(S)
    distinct = c2_params(16)
    eng.set_params_each([distinct[s % len(distinct)] for s in range(S)])

    def do_chan():
        chan.process_device(capture.data_ptr(), iq.data_ptr(), T, stream=sp)

    def do_chain():
        eng.process_device(iq.data_ptr(), audio.data_ptr(), T, row_every=T, spec_ptr=spec.data_ptr(),
                           wf_ptr=wf.data_ptr(), cuda_stream=sp)

    def timed(fn):
        for _ in range(a.warmup):
            fn()
        stream.synchronize()
        ms = []
        for _ in range(a.calls):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            fn()
            e1.record(stream)
            e1.synchronize()
            ms.append(e0.elapsed_time(e1))
        return float(np.median(ms)), float(np.min(ms)), float(np.max(ms))

    t_chan = timed(do_chan)
    t_chain = timed(do_chain)
    t_both = timed(lambda: (do_chan(), do_chain()))
    t_shift = None
    r = np.random.Generator(np.random.PCG64(2025))
    shifts = r.integers(1, 96001, S) * r.choice([-1, 1], S)
    if a.shift:
        chan.set_shift(shifts)
        t_shift = timed(do_chan)
    chan.synchronize()
    t_real = t_real_shift = None
    if a.real:
        M_real = 2 * M
        n_cap_real = T * rx.BLOCK * M_real // 2
        capture_real = torch.randint(-3277, 3278, (n_cap_real,), generator=g, device=dev, dtype=torch.int16)
        chan_real = rx.Channelizer(M_real, S, real=True)
        chan_real.set_map([(r // 2) % M for r in range(S)])

        def do_real():
            chan_real.process_device(capture_real.data_ptr(), iq.data_ptr(), T, stream=sp)

        t_real = timed(do_real)
        if a.shift:
            chan_real.set_shift(shifts)
            t_real_shift = timed(do_real)
        chan_real.synchronize()
        chan_real.close()
    t_q15 = t_q15_shift = t_conv = None
    if a.q15:
        capture_q15 = torch.randint(-3277, 3278, (n_cap, 2), generator=g, device=dev, dtype=torch.int16)
        capture_conv = torch.empty((n_cap, 2), dtype=torch.float32, device=dev)
        chan_q15 = rx.Channelizer(M, S, q15=True)
        chan_q15.set_map([(r // 2) % M for r in range(S)])
        chan_conv = rx.Channelizer(M, S)
        chan_conv.set_map([(r // 2) % M for r in range(S)])

        def do_q15():
            chan_q15.process_device(capture_q15.data_ptr(), iq.data_ptr(), T, stream=sp)

        def do_conv():
            with torch.cuda.stream(stream):
                torch.mul(capture_q15, 1.0 / 32768.0, out=capture_conv)
            chan_conv.process_device(capture_conv.data_ptr(), iq.data_ptr(), T, stream=sp)

        t_q15 = timed(do_q15)
        t_conv = timed(do_conv)
        if a.shift:
            chan_q15.set_shift(shifts)
            t_q15_shift = timed(do_q15)
        for c in (chan_q15, chan_conv):
            c.synchronize()
            c.close()
    rates = rate_table(g, dev, iq, sp, timed, shifts, S, T) if a.rates else None
    diversity = diversity_table(g, dev, iq, sp, timed, shifts, S, T, a.diversity) if a.diversity else None
    image = image_table(g, dev, iq, sp, timed, shifts, S, T) if a.image else None
    eng.synchronize()
    bytes_moved = n_cap * 8 + S * T * rx.BLOCK * 8
    res = {
        "card": card(),
        "shape": {"channels": M, "receivers": S, "receivers_per_channel": S // M, "blocks_per_call": T,
                  "capture_msps": M * 96e3 / 1e6, "capture_bytes": n_cap * 8, "iq_bytes": S * T * rx.BLOCK * 8},
        "calls": a.calls, "warmup": a.warmup,
        "chan_ms": {"median": t_chan[0], "min": t_chan[1], "max": t_chan[2]},
        "chain_c2_ms": {"median": t_chain[0], "min": t_chain[1], "max": t_chain[2]},
        "chan_plus_chain_ms": {"median": t_both[0], "min": t_both[1], "max": t_both[2]},
        "chan_capture_msps": n_cap / (t_chan[0] * 1e-3) / 1e6,
        "chan_receiver_blocks_per_s": S * T / (t_chan[0] * 1e-3),
        "chan_bytes_moved": bytes_moved,
        "chan_hbm_share_of_7p7_tbs": bytes_moved / (t_chan[0] * 1e-3) / HBM_BYTES_PER_S,
        "chan_over_chain": t_chan[0] / t_chain[0],
        "goal_chan_le_25pct_of_chain": t_chan[0] <= 0.25 * t_chain[0],
    }
    if t_shift:
        res["chan_all_shifted_ms"] = {"median": t_shift[0], "min": t_shift[1], "max": t_shift[2]}
        res["shift_overhead"] = t_shift[0] / t_chan[0] - 1.0
        res["goal_shift_overhead_le_10pct"] = t_shift[0] <= 1.10 * t_chan[0]
    if t_real:
        real_bytes = n_cap_real * 2 + S * T * rx.BLOCK * 8
        res["real"] = {"channels": M_real, "capture_msps": M_real * 96e3 / 1e6, "capture_bytes": n_cap_real * 2,
                       "chan_ms": {"median": t_real[0], "min": t_real[1], "max": t_real[2]},
                       "bytes_moved": real_bytes,
                       "hbm_share_of_7p7_tbs": real_bytes / (t_real[0] * 1e-3) / HBM_BYTES_PER_S,
                       "over_complex": t_real[0] / t_chan[0],
                       "goal_le_1p1_of_complex": t_real[0] <= 1.10 * t_chan[0]}
        if t_real_shift:
            res["real"]["all_shifted_ms"] = {"median": t_real_shift[0], "min": t_real_shift[1], "max": t_real_shift[2]}
            res["real"]["shift_overhead"] = t_real_shift[0] / t_real[0] - 1.0
    if t_q15:
        iq_bytes = S * T * rx.BLOCK * 8
        q15_bytes = n_cap * 4 + iq_bytes
        conv_bytes = n_cap * 4 + n_cap * 8 + bytes_moved     # int16 read, float written, then the float call
        res["q15"] = {"capture_bytes": n_cap * 4,
                      "chan_ms": {"median": t_q15[0], "min": t_q15[1], "max": t_q15[2]},
                      "bytes_moved": q15_bytes,
                      "hbm_share_of_7p7_tbs": q15_bytes / (t_q15[0] * 1e-3) / HBM_BYTES_PER_S,
                      "over_float": t_q15[0] / t_chan[0],
                      "goal_le_float": t_q15[0] <= t_chan[0],
                      "convert_plus_float_ms": {"median": t_conv[0], "min": t_conv[1], "max": t_conv[2]},
                      "convert_plus_float_bytes_moved": conv_bytes,
                      "convert_plus_float_hbm_share_of_7p7_tbs": conv_bytes / (t_conv[0] * 1e-3) / HBM_BYTES_PER_S}
        if t_q15_shift:
            res["q15"]["all_shifted_ms"] = {"median": t_q15_shift[0], "min": t_q15_shift[1], "max": t_q15_shift[2]}
            res["q15"]["shift_overhead"] = t_q15_shift[0] / t_q15[0] - 1.0
    if rates:
        res["rates"] = rates
    if diversity:
        res["diversity"] = {"n_inputs": a.diversity, "every_receiver_shifted_and_weighted": True, **diversity}
    if image:
        res["image"] = {"every_receiver_shifted": True, **image}
    print(json.dumps(res, indent=1))
    if a.json:
        with open(a.json, "w") as f:
            json.dump(res, f, indent=1)
    chan.close()
    eng.close()


if __name__ == "__main__":
    main()
