"""GPU tier: the CUDA path, called through the C-ABI (libt41rx.so), against the CPU oracle.

 * bit-exact kernel, exact oscillator (T41RX_FLAG_EXACT_NCO): every output and every piece of
   debug state is BIT-IDENTICAL to the oracle on all cases (C1-C5 scaled down + edge cases), and
   the audio digests equal the golden vectors the reference itself produced;
 * bit-exact kernel, closed-form FP64 oscillator (T41RX_FLAG_PHASED_KERNEL): audio SNR > 120 dB
   with > 99.9 % of samples bit-identical;
 * default = throughput kernel (FP32 with FMA contraction, blocked-scan recurrences; SAM receivers
   stay on the bit-exact kernel): the tolerance the north star states -- audio SNR >= 90 dB
   (measured: > 100 dB), spectrum rows within 1 LSB and >= 99.9 % identical, PSK31 bits /
   characters and AGC / mode state transitions identical (rx_driver.assert_within_tolerance);
 * at BASELINE.json's full sizes: size-independent properties (call-chunking invariance,
   receiver permutation invariance, replicated receivers agree) plus oracle spot checks.
"""
import hashlib
import os

import numpy as np
import pytest

import cases
import oracle_py as O
import rx_driver
from t41_sdr_b200 import rx, synth

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_vectors.npz")


def _receiver(n):
    # fails loudly (T41RxError) if the CUDA library or the device is unusable
    return rx.Receiver(n)


@pytest.mark.parametrize("make", cases.ALL_CASES, ids=lambda m: m.__name__)
def test_exact_mode_is_bit_identical_to_oracle(make):
    case = make()
    want = cases.run_case_on(case, lambda p: O.OracleStream(p))
    with _receiver(case.n_streams) as eng:
        got = rx_driver.run_case_batched(case, eng, flags=rx.FLAG_EXACT_NCO)
        # the chain as front | serial | back kernels per call (calls of 16 blocks or more: a pipeline of two time chunks,
        # rx_api.cu LaunchExact), plus the audio-spectrum by-product kernel when the call has row-producing blocks
        assert eng.kernel_launches() == sum(3 * (2 if n >= 16 else 1) + (1 if case.row_every > 0 else 0)
                                            for _, n in case.segments)
    rx_driver.assert_identical(case, got, want)


@pytest.mark.parametrize("make", cases.ALL_CASES, ids=lambda m: m.__name__)
def test_exact_mode_fused_kernel_is_bit_identical_too(make):
    """T41RX_FLAG_FUSED_EXACT: the same chain as ONE kernel (serial stages on one lane per receiver)."""
    case = make()
    want = cases.run_case_on(case, lambda p: O.OracleStream(p))
    with _receiver(case.n_streams) as eng:
        got = rx_driver.run_case_batched(case, eng, flags=rx.FLAG_EXACT_NCO | rx.FLAG_FUSED_EXACT)
        assert eng.kernel_launches() == len(case.segments) * (2 if case.row_every > 0 else 1)
    rx_driver.assert_identical(case, got, want)


@pytest.mark.parametrize("make", cases.ALL_CASES, ids=lambda m: m.__name__)
def test_exact_mode_matches_reference_golden(make):
    golden = np.load(GOLDEN)
    case = make()
    with _receiver(case.n_streams) as eng:
        got = rx_driver.run_case_batched(case, eng, flags=rx.FLAG_EXACT_NCO)
    for s, r in enumerate(got):
        key = "%s/%d/" % (case.name, s)
        audio = r["audio"].copy()
        if np.isnan(audio).any():
            continue  # NaN payloads are implementation defined; covered by the oracle comparison
        assert hashlib.sha256(audio.tobytes()).hexdigest() == bytes(golden[key + "audio_sha256"]).hex(), key
        assert np.array_equal(r["spec"], golden[key + "spec"]), key
        assert np.array_equal(r["wf"], golden[key + "wf"]), key
        if case.row_every > 0:
            rx_driver._check_audio_spec(key, r, dict(audio_ypixel=golden[key + "audio_ypixel"],
                                                     audio_max_sq_ave=golden[key + "audio_max_sq_ave"],
                                                     spec_frames=golden[key + "spec_frames"],
                                                     audio_frames=golden[key + "audio_frames"],
                                                     spec=golden[key + "spec"]), exact_max=True)
        if case.psk:
            assert np.array_equal(r["psk_bits"], golden[key + "psk_bits"]), key
            assert np.array_equal(r["psk_chars"], golden[key + "psk_chars"]), key


def _drop_nan_receivers(case, got, want):
    if case.name == "edge_silence_fullscale":
        # NaN audio (0/0 in the NFM discriminator on silence) has no SNR: compare the rest
        keep = [i for i, w in enumerate(want) if not np.isnan(w["audio"]).any()]
        return [got[i] for i in keep], [want[i] for i in keep]
    return got, want


@pytest.mark.parametrize("make", cases.ALL_CASES, ids=lambda m: m.__name__)
def test_phased_kernel_closed_form_nco(make):
    case = make()
    want = cases.run_case_on(case, lambda p: O.OracleStream(p))
    with _receiver(case.n_streams) as eng:
        got = rx_driver.run_case_batched(case, eng, flags=rx.FLAG_PHASED_KERNEL)
    got, want = _drop_nan_receivers(case, got, want)
    stats = rx_driver.assert_within_tolerance(case, got, want, min_snr_db=90.0)
    assert min(snr for snr, _ in stats) >= 120.0
    assert min(frac for _, frac in stats) >= 0.999


@pytest.mark.parametrize("make", cases.ALL_CASES, ids=lambda m: m.__name__)
def test_default_mode_within_stated_tolerance(make):
    """flags = 0: the throughput kernel (+ the rows kernel; SAM receivers on the bit-exact kernel).
    Stated tolerance: audio SNR >= 90 dB per receiver over the run, rows within 1 LSB, discrete
    state and PSK31 output identical."""
    case = make()
    want = cases.run_case_on(case, lambda p: O.OracleStream(p))
    with _receiver(case.n_streams) as eng:
        got = rx_driver.run_case_batched(case, eng, flags=0)
    got, want = _drop_nan_receivers(case, got, want)
    stats = rx_driver.assert_within_tolerance(case, got, want, min_snr_db=90.0)
    # measured margin over the stated 90 dB (the CW low-passes remove most of their two-tone input: the same absolute
    # error weighs more in what is left, 92 dB at worst)
    assert min(snr for snr, _ in stats) >= (90.0 if case.name == "c8_cw_filters" else 100.0)


def test_lms_notch_on_the_throughput_kernel():
    """T41RX_FLAG_FAST_LMS: the automatic notch / LMS noise reduction as one warp's cooperative LMS inside the
    throughput kernel.  The notch cancels most of its input, so the same FP32 re-ordering error weighs 20-30 dB
    more in its output: the stated bound for this opt-in path is 70 dB (measured 75-117 dB); discrete state of the
    rest of the chain identical."""
    case = cases.c7_lms_notch()
    want = cases.run_case_on(case, lambda p: O.OracleStream(p))
    with _receiver(case.n_streams) as eng:
        got = rx_driver.run_case_batched(case, eng, flags=rx.FLAG_FAST_LMS)
    stats = rx_driver.assert_within_tolerance(case, got, want, min_snr_db=70.0)
    assert max(s for s, _ in stats) > 100.0


def test_sam_on_the_throughput_kernel():
    """T41RX_FLAG_FAST_SAM: the SAM PLL as one serial lane inside the throughput kernel.  While the loop pulls in
    (carrier offsets of up to 200 Hz against a ~30 Hz loop: 10-15 blocks here) it is chaotic - ApproxAtan2 returns
    +-2 pi where pi / 2 is meant (Demod.cpp:148-197) - and a 1e-7 difference at its input gives another transient;
    once locked the trajectories coincide again: >= 90 dB (measured 120-136 dB) from block 16 on.  Everything in
    front of the detector (AGC state, RFgain, ...) is identical throughout; the NFM half of the case is untouched."""
    case = cases.c3_nfm_sam_agc()
    want = cases.run_case_on(case, lambda p: O.OracleStream(p))
    with _receiver(case.n_streams) as eng:
        got = rx_driver.run_case_batched(case, eng, flags=rx.FLAG_FAST_SAM)
        assert eng.kernel_launches() == 3 * len(case.segments)     # rows + stream + by-products: no bit-exact kernel
    n_sam = 0
    for s_, (g, w) in enumerate(zip(got, want)):
        mode = case.segments[0][0][s_].mode
        ga, wa = g["audio"], w["audio"]
        if mode == cases.SAM:
            n_sam += 1
            assert O.snr_db(wa[16:], ga[16:]) >= 90.0, (s_, O.snr_db(wa[16:], ga[16:]))
        else:
            ok = ~(np.isnan(ga) | np.isnan(wa))
            assert O.snr_db(np.where(ok, wa, 0), np.where(ok, ga, 0)) >= 90.0, s_
        for f in cases.DEBUG_INT_FIELDS:
            assert getattr(g["debug"], f) == getattr(w["debug"], f), (s_, f)
        assert np.abs(g["spec"].astype(int) - w["spec"].astype(int)).max() <= 1
    assert n_sam >= 2


def test_psk31_text_is_decoded():
    case = cases.c5_psk31()
    with _receiver(case.n_streams) as eng:
        got = rx_driver.run_case_batched(case, eng, flags=0)
    for r in got:
        chars = bytes(r["psk_chars"][r["psk_chars"] > 0])
        assert cases.PSK_TEXT.encode() in chars


def _float_to_q15(x):
    """arm_float_to_q15 (oracle/cmsis_port.c): saturate(trunc(x * 32768)); NaN -> 0 (the target's VCVT)"""
    v = x.astype(np.float32) * np.float32(32768.0)
    q = np.where(np.isnan(v), 0.0, np.clip(np.trunc(v.astype(np.float64)), -2147483648.0, 2147483647.0))
    return np.clip(q, -32768, 32767).astype(np.int16)


def test_q15_entry_point_is_the_firmware_block_format():
    """t41rx_process_q15: q15 I/Q in, q15 audio out (Process.cpp:102-111, 936-937).  The synthetic I/Q of the
    parity cases IS q15 / 32768, so the oracle on the float input is the reference for the q15 call."""
    case = cases.c2_ssb_am_mix()
    want = cases.run_case_on(case, lambda p: O.OracleStream(p))
    iq = np.stack(case.iq)
    iq16 = np.round(iq * 32768.0).astype(np.int16)
    assert np.array_equal(iq16.astype(np.float32) / np.float32(32768.0), iq)
    params = [rx_driver.to_rx_params(p) for p in case.segments[0][0]]
    with _receiver(case.n_streams) as eng:
        eng.set_params_each(params)
        exact = eng.process_q15(iq16, row_every=case.row_every, flags=rx.FLAG_EXACT_NCO)
    with _receiver(case.n_streams) as eng:
        eng.set_params_each(params)
        fast = eng.process_q15(iq16, row_every=case.row_every, flags=0)
    for s_, w in enumerate(want):
        ref16 = _float_to_q15(w["audio"])
        assert np.array_equal(exact["audio"][s_], ref16), s_                # bit-exact kernel: identical q15 words
        assert np.array_equal(exact["spec"][s_], w["spec"])
        d = np.abs(fast["audio"][s_].astype(np.int32) - ref16.astype(np.int32))
        assert d.max() <= 1 and np.mean(d == 0) >= 0.99, (s_, int(d.max()), float(np.mean(d == 0)))
        assert np.array_equal(fast["spec"][s_], w["spec"])


def test_audio_spectrum_by_product_entry_points():
    """The audio-spectrum / S-meter by-product (Process.cpp:550-570) through the three entry points: host float,
    host q15 and device pointers give the same rows; unbinding stops the output; the S-meter helper matches the
    oracle's restatement of Display.cpp:980."""
    torch = pytest.importorskip("torch")
    case = cases.c2_ssb_am_mix()
    want = cases.run_case_on(case, lambda p: O.OracleStream(p))
    iq = np.stack(case.iq)
    S, T = iq.shape[:2]
    R = (T + case.row_every - 1) // case.row_every
    params = [rx_driver.to_rx_params(p) for p in case.segments[0][0]]
    outs = []
    for flags in (rx.FLAG_EXACT_NCO, 0):
        with _receiver(S) as eng:
            eng.set_params_each(params)
            host = eng.process(iq, row_every=case.row_every, flags=flags, want_audio_spec=True)
        with _receiver(S) as eng:
            eng.set_params_each(params)
            q15 = eng.process_q15(np.round(iq * 32768.0).astype(np.int16), row_every=case.row_every, flags=flags,
                                  want_audio_spec=True)
        with _receiver(S) as eng:
            eng.set_params_each(params)
            d_iq = torch.from_numpy(iq).cuda()
            d_audio = torch.empty((S, T, 2048), dtype=torch.float32, device="cuda")
            d_pix = torch.full((S, R, rx.AUDIO_SPEC_PIXELS), -7, dtype=torch.int32, device="cuda")
            d_max = torch.full((S, R), -7.0, dtype=torch.float32, device="cuda")
            d_spec = torch.zeros((S, R, 512), dtype=torch.int16, device="cuda")
            d_sfr = torch.full((S, R, rx.SPEC_FRAME_BYTES), 9, dtype=torch.uint8, device="cuda")
            d_afr = torch.full((S, R, rx.AUDIO_SPEC_PIXELS), 9, dtype=torch.uint8, device="cuda")
            eng.bind_audio_spectrum(d_pix.data_ptr(), d_max.data_ptr())
            eng.bind_control_frames(d_sfr.data_ptr(), d_afr.data_ptr())
            with pytest.raises(rx.T41RxError):        # the spectrum frame needs the spectrum rows
                eng.process_device(d_iq.data_ptr(), d_audio.data_ptr(), T, row_every=case.row_every, flags=flags)
            eng.process_device(d_iq.data_ptr(), d_audio.data_ptr(), T, row_every=case.row_every,
                               spec_ptr=d_spec.data_ptr(), flags=flags)
            eng.synchronize()
            eng.bind_audio_spectrum(None, None)
            eng.bind_control_frames(None, None)
            dev_pix, dev_max = d_pix.cpu().numpy(), d_max.cpu().numpy()
            assert np.array_equal(d_sfr.cpu().numpy(), host["spec_frames"])
            assert np.array_equal(d_afr.cpu().numpy(), host["audio_frames"])
            # unbound: a second call leaves the buffers alone
            d_pix.fill_(-7)
            eng.process_device(d_iq.data_ptr(), d_audio.data_ptr(), T, row_every=case.row_every, flags=flags)
            eng.synchronize()
            assert int(d_pix.max()) == -7
        for o in (q15,):
            assert np.array_equal(o["spec_frames"], host["spec_frames"]) and np.array_equal(o["audio_frames"], host["audio_frames"])
            assert np.array_equal(o["audio_ypixel"], host["audio_ypixel"])
            assert np.array_equal(o["audio_max_sq_ave"].view(np.uint32), host["audio_max_sq_ave"].view(np.uint32))
        assert np.array_equal(dev_pix, host["audio_ypixel"])
        assert np.array_equal(dev_max.view(np.uint32), host["audio_max_sq_ave"].view(np.uint32))
        for s_, w in enumerate(want):
            rx_driver._check_audio_spec("receiver %d flags %d" % (s_, flags),
                                        dict(audio_ypixel=host["audio_ypixel"][s_], audio_max_sq_ave=host["audio_max_sq_ave"][s_],
                                             spec_frames=host["spec_frames"][s_], audio_frames=host["audio_frames"][s_],
                                             spec=host["spec"][s_]),
                                        w, exact_max=(flags != 0))
        outs.append(host)
    lib = O.tier_b()
    for v in outs[0]["audio_max_sq_ave"].ravel()[:8]:
        assert rx.smeter_dbm(float(v), -2.0, 3, 1) == lib.t41o_smeter_dbm(float(v), -2.0, 3, 1)


def test_error_codes():
    with _receiver(3) as eng:
        with pytest.raises(rx.T41RxError):
            eng.set_params(rx_driver.to_rx_params(cases.P(mode=4)))
        with pytest.raises(rx.T41RxError):
            eng.set_params(rx.default_params(), first=2, count=5)
        with pytest.raises(ValueError):
            eng.process(np.zeros((2, 1, 2048, 2), np.float32))


# ---------------- BASELINE sizes: properties + spot checks ----------------
def _c2_bank(n_streams, n_blocks, n_distinct=16):
    """C2-shaped bank: even receivers USB, odd AM, per-receiver NCO; the I/Q of receiver s is
    distinct signal (s % n_distinct), so a large bank needs little host memory to build."""
    r = np.random.Generator(np.random.PCG64(2024))
    base_p, base_iq = [], []
    for k in range(n_distinct):
        nco = int(r.integers(-20000, 20001))
        if k % 2 == 0:
            base_p.append(cases.P(mode=cases.USB, f_lo_cut=300, f_hi_cut=3000, nco_freq=nco))
            base_iq.append(synth.tone(900 + k, n_blocks, float(r.uniform(300, 2700)), mode=cases.USB, nco_freq=nco))
        else:
            base_p.append(cases.P(mode=cases.AM, nco_freq=nco))
            base_iq.append(synth.am(900 + k, n_blocks, mode=cases.AM, nco_freq=nco))
    params = [rx_driver.to_rx_params(base_p[s % n_distinct]) for s in range(n_streams)]
    iq = np.stack([base_iq[s % n_distinct] for s in range(n_streams)])
    return base_p, base_iq, params, iq


def test_c2_full_size_1024_receivers():
    S, T, D = 1024, 16, 16
    base_p, base_iq, params, iq = _c2_bank(S, T, D)
    with _receiver(S) as eng:
        eng.set_params_each(params)
        one = eng.process(iq, row_every=T)
    audio = one["audio"]
    # replicated receivers (same params, same input) agree exactly wherever they sit in the grid
    for k in range(D):
        grp = audio[k::D]
        assert np.array_equal(grp.view(np.uint32), np.broadcast_to(grp[0], grp.shape).view(np.uint32))
        assert np.array_equal(one["spec"][k::D], np.broadcast_to(one["spec"][k], one["spec"][k::D].shape))
    # spot check against the oracle (default mode tolerance)
    for k in range(D):
        w = O.OracleStream(base_p[k]).process(base_iq[k], T)
        assert O.snr_db(w["audio"], audio[k]) >= 100.0
        assert np.abs(w["spec"].astype(int) - one["spec"][k].astype(int)).max() <= 1
    # call-chunking invariance: 16 blocks at once == 5 + 11 blocks (state hand-over through HBM)
    with _receiver(S) as eng:
        eng.set_params_each(params)
        a = eng.process(iq[:, :5])["audio"]
        b = eng.process(iq[:, 5:])["audio"]
    assert np.array_equal(np.concatenate([a, b], axis=1).view(np.uint32), audio.view(np.uint32))
    # receiver permutation invariance: no cross-talk between receivers
    perm = np.random.Generator(np.random.PCG64(7)).permutation(S)
    with _receiver(S) as eng:
        eng.set_params_each([params[i] for i in perm])
        p = eng.process(iq[perm])["audio"]
    assert np.array_equal(p.view(np.uint32), audio[perm].view(np.uint32))


def test_host_pipeline_chunking_is_invisible():
    """t41rx_process cuts a long call into launches over block ranges (copy / compute / copy-back pipeline); the
    result must be the one launch of t41rx_process_device, bit for bit: audio, rows whose period (5) does not
    divide the chunk length (4), by-products, PSK31 bits, end state."""
    torch = pytest.importorskip("torch")
    S, T, D, every = 64, 64, 16, 5
    base_p, base_iq, params, iq = _c2_bank(S, T, D)
    for p in params:
        p.psk31_enable = 1
        p.spectrum_zoom = 2
    R = (T + every - 1) // every
    with _receiver(S) as eng:
        eng.set_params_each(params)
        n0 = eng.kernel_launches()
        host = eng.process(iq, row_every=every, want_psk=True, want_audio_spec=True)
        assert eng.kernel_launches() - n0 >= 16           # really cut into chunks
        dbg_host = [eng.debug(s) for s in (0, 1, S - 1)]
    with _receiver(S) as eng:
        eng.set_params_each(params)
        d = {k: torch.zeros(shape, dtype=dt, device="cuda") for k, shape, dt in (
            ("audio", (S, T, 2048), torch.float32), ("spec", (S, R, 512), torch.int16), ("wf", (S, R, 512), torch.int16),
            ("bits", (S, T), torch.int8), ("chars", (S, T), torch.uint8), ("pix", (S, R, rx.AUDIO_SPEC_PIXELS), torch.int32),
            ("mx", (S, R), torch.float32), ("sfr", (S, R, rx.SPEC_FRAME_BYTES), torch.uint8),
            ("afr", (S, R, rx.AUDIO_SPEC_PIXELS), torch.uint8))}
        d_iq = torch.from_numpy(iq).cuda()
        eng.bind_audio_spectrum(d["pix"].data_ptr(), d["mx"].data_ptr())
        eng.bind_control_frames(d["sfr"].data_ptr(), d["afr"].data_ptr())
        eng.process_device(d_iq.data_ptr(), d["audio"].data_ptr(), T, row_every=every, spec_ptr=d["spec"].data_ptr(),
                           wf_ptr=d["wf"].data_ptr(), psk_bits_ptr=d["bits"].data_ptr(), psk_chars_ptr=d["chars"].data_ptr())
        eng.synchronize()
        dbg_dev = [eng.debug(s) for s in (0, 1, S - 1)]
    pairs = (("audio", "audio"), ("spec", "spec"), ("wf", "wf"), ("psk_bits", "bits"), ("psk_chars", "chars"),
             ("audio_ypixel", "pix"), ("audio_max_sq_ave", "mx"), ("spec_frames", "sfr"), ("audio_frames", "afr"))
    for hk, dk in pairs:
        dev = d[dk].cpu().numpy()
        assert np.array_equal(host[hk].view(np.uint8), dev.view(np.uint8)), hk
    for a_, b_ in zip(dbg_host, dbg_dev):
        assert bytes(a_) == bytes(b_)
    assert host["spec_frames"][:, :, 0].min() == ord("F") and np.abs(host["audio"]).max() > 1e-3


@pytest.mark.parametrize("S,T", [(1, 1), (149, 3), (1037, 2), (5, 17)])
def test_ragged_bank_sizes(S, T):
    """Bank sizes that do not divide into CTAs (one receiver more than there are SMs, a prime count, a single receiver
    and a single block): every receiver's output equals what the same receiver gives in a bank of its own distinct
    signals, and the oracle's within the default tolerance."""
    D = 16
    base_p, base_iq, params, iq = _c2_bank(S, T, D)
    with _receiver(S) as eng:
        eng.set_params_each(params)
        big = eng.process(iq, row_every=1)
    n = min(S, D)
    with _receiver(n) as eng:
        eng.set_params_each(params[:n])
        small = eng.process(iq[:n], row_every=1)
    for s_ in range(S):
        k = s_ % D
        if k < n:
            assert np.array_equal(big["audio"][s_].view(np.uint32), small["audio"][k].view(np.uint32)), s_
            assert np.array_equal(big["spec"][s_], small["spec"][k]) and np.array_equal(big["wf"][s_], small["wf"][k]), s_
    for k in range(n):
        w = O.OracleStream(base_p[k]).process(base_iq[k], 1)
        assert O.snr_db(w["audio"], small["audio"][k]) >= 90.0
        assert np.array_equal(w["spec"], small["spec"][k])


def test_receivers_per_cta_invariance(monkeypatch):
    """The throughput kernel's result for a receiver must not depend on how many receivers share its CTA (which
    decides which AGC lane and which shared-memory slot it gets, and how the warps interleave): a race between the
    receiver pairs, the AGC warp and the asynchronous copies would show up here as a difference."""
    S, T, D = 296, 12, 16
    base_p, base_iq, params, iq = _c2_bank(S, T, D)
    outs = []
    for g in ("1", "2", "5", "7"):
        monkeypatch.setenv("T41RX_FAST_G", g)        # developer knob of the launcher (receivers per CTA)
        with _receiver(S) as eng:
            eng.set_params_each(params)
            outs.append(eng.process(iq, row_every=4))
    monkeypatch.delenv("T41RX_FAST_G")
    for o in outs[1:]:
        assert np.array_equal(o["audio"].view(np.uint32), outs[0]["audio"].view(np.uint32))
        assert np.array_equal(o["spec"], outs[0]["spec"])


def test_bench_dump_outputs_are_the_last_timed_step(tmp_path):
    """`bench.py --dump-outputs` on the GPU: the files hold what the last of its calls returned - the same calls (warm-up,
    the clock sampler's lead-in, the timed steps) replayed through the library give the same audio and rows bit for
    bit - and `--steps` is the number of timed steps it reports."""
    import json
    import subprocess
    import sys
    import bench
    S, T, warmup, steps = 16, 4, 1, 2
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = {k: v for k, v in os.environ.items() if not k.startswith("T41RX_")}
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--gpus", "1", "--streams", str(S), "--blocks", str(T),
                          "--steps", str(steps), "--warmup", str(warmup), "--no-e2e", "--no-cpu-baseline", "--no-q15",
                          "--no-extra-configs", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, env=env,
                         timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps and line["value"] > 0
    params, sigs = bench.workload(T)
    iq = np.stack([sigs[s % len(sigs)] for s in range(S)])
    with _receiver(S) as eng:
        eng.set_params_each([params[s % len(params)] for s in range(S)])
        for _ in range(max(3, warmup) + 3 + steps):
            want = eng.process(iq, row_every=T)
    got = {k: np.load(tmp_path / (k + ".npy")) for k in ("audio", "spec", "wf")}
    assert np.array_equal(got["audio"].view(np.uint32), want["audio"].view(np.uint32))
    assert np.array_equal(got["spec"], want["spec"].astype(np.float32))
    assert np.array_equal(got["wf"], want["wf"].astype(np.float32))
    assert np.abs(got["audio"]).max() > 0


def test_c4_full_size_16384_spectrum_rows():
    S, T, D = 16384, 2, 10
    base_p = [cases.P(spectrum_zoom=k % 5, current_scale=1 + (k // 5)) for k in range(D)]
    base_iq = [synth.two_tone(400 + k, T, f1=46500.0 - 300 * k, f2=50500.0) for k in range(D)]
    params = [rx_driver.to_rx_params(base_p[s % D]) for s in range(S)]
    iq = np.stack([base_iq[s % D] for s in range(S)])
    with _receiver(S) as eng:
        eng.set_params_each(params)
        out = eng.process(iq, row_every=1, flags=rx.FLAG_EXACT_NCO)
    for k in range(D):
        w = O.OracleStream(base_p[k]).process(base_iq[k], 1)
        assert np.array_equal(out["spec"][k::D], np.broadcast_to(w["spec"], out["spec"][k::D].shape))
        assert np.array_equal(out["wf"][k::D], np.broadcast_to(w["wf"], out["wf"][k::D].shape))


def test_rows_kernel_full_bank_rows_bit_identical_and_call_chunking():
    """The rows-only kernel (default flags) on a bank large enough for three of its CTAs to share every SM: CTAs
    that mix zoom x1 with zoomed receivers (the cascade's idle lanes run on the x1 receivers' dead tiles), every
    block a row (DC-block state carried from block to block), a partial last CTA, and the same run cut into two
    calls (the second call's first block is seeded from the buffer instead).  Rows and waterfall identical to the
    oracle's for every distinct waveform and across all replicas."""
    S, T, D = 8190, 6, 10
    base_p = [cases.P(spectrum_zoom=k % 5, current_scale=1 + (k // 5)) for k in range(D)]
    base_iq = [synth.two_tone(700 + k, T, f1=46500.0 - 300 * k, f2=50500.0) for k in range(D)]
    params = [rx_driver.to_rx_params(base_p[s % D]) for s in range(S)]
    iq = np.stack([base_iq[s % D] for s in range(S)])
    with _receiver(S) as eng:
        eng.set_params_each(params)
        one = eng.process(iq, row_every=1)
    with _receiver(S) as eng:
        eng.set_params_each(params)
        a = eng.process(np.ascontiguousarray(iq[:, :2]), row_every=1)
        b = eng.process(np.ascontiguousarray(iq[:, 2:]), row_every=1)
    for key in ("spec", "wf"):
        assert np.array_equal(np.concatenate([a[key], b[key]], axis=1), one[key])
    for k in range(D):
        w = O.OracleStream(base_p[k]).process(base_iq[k], 1)
        assert np.array_equal(one["spec"][k::D], np.broadcast_to(w["spec"], one["spec"][k::D].shape)), k
        assert np.array_equal(one["wf"][k::D], np.broadcast_to(w["wf"], one["wf"][k::D].shape)), k


def test_c3_full_size_8192_nfm_sam_state_transitions():
    S, T, D = 8192, 24, 8
    case = cases.c3_nfm_sam_agc(n=D, T=T)
    base_p, base_iq = case.segments[0][0], case.iq
    params = [rx_driver.to_rx_params(base_p[s % D]) for s in range(S)]
    iq = np.stack([base_iq[s % D] for s in range(S)])
    with _receiver(S) as eng:
        eng.set_params_each(params)
        out = eng.process(iq, flags=0)
        dbg = [eng.debug(s) for s in (0, 1, 2, 3, 4, 5, 6, 7, S - 8, S - 7, S - 2, S - 1)]
    want = cases.run_case_on(cases.Case(case.name, case.segments, case.iq), lambda p: O.OracleStream(p))
    for k in range(D):
        assert O.snr_db(want[k]["audio"], out["audio"][k]) >= 100.0
        grp = out["audio"][k::D]
        assert np.array_equal(grp.view(np.uint32), np.broadcast_to(grp[0], grp.shape).view(np.uint32))
    for d, s in zip(dbg, (0, 1, 2, 3, 4, 5, 6, 7, S - 8, S - 7, S - 2, S - 1)):
        w = want[s % D]["debug"]
        for f in cases.DEBUG_INT_FIELDS:
            assert getattr(d, f) == getattr(w, f), (s, f)


def test_c5_full_size_32768_psk31_bits():
    """32768 receivers x the full message would need ~1 TB of I/Q (SURVEY section 8(d)); the bank is
    fed with 4 distinct waveforms and processed in time slices of 6 blocks, bits compared with the
    oracle's for every distinct waveform and required to agree across all replicas."""
    S, D, SLICE = 32768, 4, 6
    case = cases.c5_psk31(n=D)
    base_p, base_iq = case.segments[0][0], case.iq
    T = base_iq[0].shape[0]
    T = min(T, 20 * SLICE)
    params = [rx_driver.to_rx_params(base_p[s % D]) for s in range(S)]
    want = [O.OracleStream(base_p[k]).process(base_iq[k][:T], 0, True) for k in range(D)]
    bits = []
    with _receiver(S) as eng:
        eng.set_params_each(params)
        for b0 in range(0, T, SLICE):
            iq = np.stack([base_iq[s % D][b0:b0 + SLICE] for s in range(D)])
            iq = np.ascontiguousarray(np.tile(iq, (S // D, 1, 1, 1)))
            bits.append(eng.process(iq, want_psk=True)["psk_bits"])
    bits = np.concatenate(bits, axis=1)
    for k in range(D):
        assert np.array_equal(bits[k::D], np.broadcast_to(want[k]["psk_bits"], bits[k::D].shape))


# ---- a bank over several devices behind the C-ABI (t41rx_create_multi; SURVEY 8(b), 8(e)) ----
def _n_gpus():
    torch = pytest.importorskip("torch")
    return torch.cuda.device_count()


def test_multi_device_bank_equals_one_context():
    """t41rx_create_multi shards a bank into contiguous receiver ranges, one single-device context and one host thread
    each.  Receivers are independent, so the sharded bank must give exactly the single context's results - audio, rows,
    PSK31 output, state - whatever the shard boundaries (here 3 shards of a ragged 13-receiver bank; all on the GPUs this
    box has, several shards per GPU when it has fewer)."""
    S, T, D = 13, 12, 16
    base_p, base_iq, params, iq = _c2_bank(S, T, D)
    for p in params:
        p.psk31_enable = 1
    with _receiver(S) as eng:
        eng.set_params_each(params)
        one = eng.process(iq, row_every=4, want_psk=True)
        dbg_one = [eng.debug(s) for s in range(S)]
    devs = [g % _n_gpus() for g in range(3)]
    with rx.MultiReceiver(S, devs) as m:
        assert [(f, c) for _, f, c in m.shards()] == [(0, 4), (4, 4), (8, 5)]
        m.set_params_each(params)
        many = m.process(iq, row_every=4, want_psk=True)
        dbg_many = [m.debug(s) for s in range(S)]
        iq16 = np.round(iq * 32768.0).astype(np.int16)
    for k in ("audio", "spec", "wf", "psk_bits", "psk_chars"):
        a, b = one[k], many[k]
        assert np.array_equal(a.view(np.uint32) if a.dtype == np.float32 else a, b.view(np.uint32) if b.dtype == np.float32 else b), k
    for a, b in zip(dbg_one, dbg_many):
        for f in cases.DEBUG_INT_FIELDS:
            assert getattr(a, f) == getattr(b, f), f
    # the q15 entry point through the same fan-out
    with _receiver(S) as eng:
        eng.set_params_each(params)
        one16 = eng.process_q15(iq16, row_every=4)
    with rx.MultiReceiver(S, devs) as m:
        m.set_params_each(params)
        many16 = m.process_q15(iq16, row_every=4)
    assert np.array_equal(one16["audio"], many16["audio"]) and np.array_equal(one16["spec"], many16["spec"])


def test_multi_device_errors_name_the_shard():
    with pytest.raises(rx.T41RxError) as e:
        rx.MultiReceiver(8, [0, 99])
    assert "shard 1" in str(e.value) and "device" in str(e.value)
    with rx.MultiReceiver(8, [0, 0]) as m:
        p = rx.default_params()
        p.agc_mode = 77
        with pytest.raises(rx.T41RxError):
            m.set_params(p, first=3, count=3)


def test_multi_device_resident_and_row_gather():
    """Device-resident fan-out (per-shard device pointers) and the optional gather of spectrum rows to the first device:
    NCCL send / recv when the shards sit on distinct GPUs, peer / device copies otherwise.  The gathered rows must be the
    single context's rows in receiver order."""
    torch = pytest.importorskip("torch")
    S, T, D = 16, 8, 16
    base_p, base_iq, params, iq = _c2_bank(S, T, D)
    with _receiver(S) as eng:
        eng.set_params_each(params)
        one = eng.process(iq, row_every=4)
    n_gpu = _n_gpus()
    devs = [0, 1] if n_gpu >= 2 else [0, 0]
    R = 2
    with rx.MultiReceiver(S, devs) as m:
        m.set_params_each(params)
        bufs = []
        for dev, first, count in m.shards():
            d = torch.device("cuda", dev)
            bufs.append(dict(iq=torch.from_numpy(iq[first:first + count]).to(d),
                             audio=torch.zeros((count, T, 2048), dtype=torch.float32, device=d),
                             spec=torch.zeros((count, R, 512), dtype=torch.int16, device=d),
                             wf=torch.zeros((count, R, 512), dtype=torch.int16, device=d)))
        for dev in set(devs):
            torch.cuda.synchronize(dev)
        m.process_device([b["iq"].data_ptr() for b in bufs], [b["audio"].data_ptr() for b in bufs], T, 4,
                         [b["spec"].data_ptr() for b in bufs], [b["wf"].data_ptr() for b in bufs])
        m.synchronize()
        audio = np.concatenate([b["audio"].cpu().numpy() for b in bufs])
        assert np.array_equal(audio.view(np.uint32), one["audio"].view(np.uint32))
        dst = torch.zeros((S, R, 512), dtype=torch.int16, device=torch.device("cuda", devs[0]))
        used_nccl = m.gather_rows([b["spec"].data_ptr() for b in bufs], R * 512 * 2, dst.data_ptr())
        assert np.array_equal(dst.cpu().numpy(), one["spec"])
        assert used_nccl == (n_gpu >= 2)
