"""CPU tier, part 2: the product's host side, without a GPU.

 * libt41rx.so loads and exports every entry point include/t41rx.h declares.
 * The control path (filter / AGC / zoom design in C++) produces tables bit-identical to the
   oracle's, including the sticky AGC tuning across mode changes.
 * Without a CUDA device the library refuses to work (no CPU fallback).
 * The kernel's phase functions, compiled for the host by tests/devtools (a development aid
   that is not part of the product), reproduce the oracle bit for bit: this checks index
   arithmetic, shared-memory overlays and state hand-over before GPU time is spent.
"""
import ctypes as C
import os
import re

import numpy as np
import pytest

import cases
import oracle_py as O
import rx_driver
from t41_sdr_b200 import rx

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _have_gpu():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def test_library_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "t41rx.h")).read()
    declared = sorted(set(re.findall(r"\b(t41rx_[a-z_0-9]+)\s*\(", header)))
    assert len(declared) >= 18
    L = rx.lib()
    for name in declared:
        assert hasattr(L, name), "libt41rx.so does not export %s" % name
    assert set(declared) == set(rx.EXPORTS)
    assert b"sm_100a" in L.t41rx_version()


def test_params_struct_layout_is_shared():
    assert C.sizeof(rx.Params) == C.sizeof(O.Params) == (18 + 1 + 14 + 2 + 2 + 1) * 4
    assert [f[0] for f in rx.Params._fields_] == [f[0] for f in O.Params._fields_]
    a, b = rx.default_params(), O.default_params()
    assert bytes(a) == bytes(b)
    for mode in (0, 1, 2, 3, 5, 8):
        assert rx.mode_default_cuts(mode) == O.mode_default_cuts(mode)


SEQUENCES = {
    "defaults": [],
    "usb_2k7": [cases.P(mode=cases.USB, f_lo_cut=300, f_hi_cut=3000)],
    "lsb": [cases.P(mode=cases.LSB)],
    "am_wide": [cases.P(mode=cases.AM, f_lo_cut=-5000, f_hi_cut=5000, agc_mode=2, agc_thresh=30)],
    "nfm": [cases.P(mode=cases.NFM, nfm_filter_bw=9000, agc_mode=4)],
    "sticky_hang_thresh": [cases.P(agc_mode=3), cases.P(agc_mode=1)],          # B12
    "agc_off_then_slow": [cases.P(agc_mode=0), cases.P(agc_mode=2, agc_thresh=10)],
    "zoom16_psk": [cases.P(spectrum_zoom=4, f_lo_cut=-100, f_hi_cut=100, psk31_enable=1)],
    "clamped_10k": [cases.P(mode=cases.AM, f_lo_cut=-11000, f_hi_cut=11000, spectrum_zoom=0)],
}


@pytest.mark.parametrize("name", sorted(SEQUENCES))
def test_control_path_tables_equal_oracle(name):
    seq = SEQUENCES[name]
    o = O.OracleStream()
    for p in seq:
        o.set_params(p)
    if seq and seq[-1].mode == cases.NFM:
        # the firmware re-designs the decimators for nfmFilterBW at the top of every NFM block
        # (Process.cpp:259); the product carries those taps from set_params on
        o.process(np.zeros((1, 2048, 2), np.float32))
    want = o.tables()
    got = rx.design_tables([rx_driver.to_rx_params(p) for p in seq])
    for k, v in want.items():
        if isinstance(v, np.ndarray):
            assert np.array_equal(v.view(np.uint32), got[k].view(np.uint32)), "%s: table %s differs" % (name, k)
        else:
            assert v == got[k], "%s: %s" % (name, k)


def test_invalid_parameters_are_rejected():
    bad = [cases.P(mode=4), cases.P(agc_mode=7), cases.P(spectrum_zoom=5), cases.P(f_lo_cut=3000, f_hi_cut=200),
           cases.P(audio_volume=101), cases.P(current_scale=-1)]
    for p in bad:
        with pytest.raises(rx.T41RxError):
            rx.design_tables([rx_driver.to_rx_params(p)])
        with pytest.raises(ValueError):
            O.OracleStream().set_params(p)
    # rfGainAllBands: the product accepts +-40 dB (t41rx.h T41RX_RF_GAIN_ALL_BANDS_MAX; the reference has no bound, but
    # larger steps between calls take the throughput kernel below its tolerance, and from about -760 dB the FP32 gain
    # rounds to 0 and the kernel's DC-block state became 0 / 0)
    for g in (-41, 41, -200, 200, -1000, -2 ** 31, 2 ** 31 - 1):
        with pytest.raises(rx.T41RxError):
            rx.design_tables([rx_driver.to_rx_params(cases.P(rf_gain_all_bands=g))])
    for g in (-40, 40):
        rx.design_tables([rx_driver.to_rx_params(cases.P(rf_gain_all_bands=g))])


@pytest.mark.skipif(_have_gpu(), reason="checks the no-GPU behaviour")
def test_no_gpu_means_failure_not_fallback():
    with pytest.raises(rx.T41RxError) as e:
        rx.Receiver(4)
    assert "no CUDA device" in str(e.value) or "CUDA" in str(e.value)


# ---- kernel phase logic on the host (development aid, see tests/devtools/kernel_emul.cpp) ----
EMUL_CASES = [cases.c1_single_usb_agc_off, cases.c2_ssb_am_mix, cases.c3_nfm_sam_agc, cases.c4_zoom_rows, cases.c6_receive_eq, cases.c7_lms_notch, cases.c8_cw_filters, cases.c9_kim_spectral_nb,
              cases.edge_silence_fullscale, cases.edge_param_changes]


@pytest.mark.parametrize("make", EMUL_CASES, ids=lambda m: m.__name__)
def test_kernel_phases_emulated_exact(make):
    case = make()
    want = cases.run_case_on(case, lambda p: O.OracleStream(p))
    eng = rx_driver.EmulReceiver(case.n_streams)
    got = rx_driver.run_case_batched(case, eng, flags=rx.FLAG_EXACT_NCO)
    eng.close()
    rx_driver.assert_identical(case, got, want)


@pytest.mark.parametrize("make", [cases.c2_ssb_am_mix, cases.edge_param_changes, cases.c5_psk31],
                         ids=lambda m: m.__name__)
def test_kernel_phases_emulated_closed_form_nco(make):
    case = make()
    want = cases.run_case_on(case, lambda p: O.OracleStream(p))
    eng = rx_driver.EmulReceiver(case.n_streams)
    got = rx_driver.run_case_batched(case, eng, flags=0)
    eng.close()
    stats = rx_driver.assert_within_tolerance(case, got, want, min_snr_db=120.0)
    assert min(f for _, f in stats) > 0.999      # almost every sample is bit-identical


EMUL_SPLIT_ROWS = 0x100   # tests/devtools/kernel_emul.cpp: rows through the rows-only schedule


@pytest.mark.parametrize("make", [cases.c1_single_usb, cases.c3_nfm_sam_agc, cases.c4_zoom_rows,
                                  cases.edge_param_changes], ids=lambda m: m.__name__)
def test_rows_only_schedule_emulated(make):
    """The rows-only schedule (what t41rx_rows_kernel runs beside the throughput kernel: DC-block state
    seeded from the previous block's tail, RFgain extrapolated from the launch-start state) must give
    the oracle's spectrum and waterfall rows bit for bit, and leave the rest of the chain untouched."""
    case = make()
    want = cases.run_case_on(case, lambda p: O.OracleStream(p))
    eng = rx_driver.EmulReceiver(case.n_streams)
    got = rx_driver.run_case_batched(case, eng, flags=rx.FLAG_EXACT_NCO | EMUL_SPLIT_ROWS)
    eng.close()
    rx_driver.assert_identical(case, got, want)


EMUL_SPLIT_EXACT = 0x200  # tests/devtools/kernel_emul.cpp: the chain as the front | serial | back kernels


@pytest.mark.parametrize("make", EMUL_CASES + [cases.c5_psk31, cases.c1_single_usb], ids=lambda m: m.__name__)
def test_split_exact_kernels_emulated(make):
    """The bit-exact chain as the product runs it by default (t41rx_exact_front_kernel, t41rx_exact_serial_kernel with
    thread = receiver, t41rx_exact_back_kernel; hand-over through receiver-minor scratch) must equal the oracle bit for
    bit on every output and every piece of state, like the fused schedule: every mode, AGC on / off, equaliser, LMS /
    notch, CW filters, parameter changes between calls, silence and full scale."""
    case = make()
    want = cases.run_case_on(case, lambda p: O.OracleStream(p))
    eng = rx_driver.EmulReceiver(case.n_streams)
    got = rx_driver.run_case_batched(case, eng, flags=rx.FLAG_EXACT_NCO | EMUL_SPLIT_EXACT)
    eng.close()
    rx_driver.assert_identical(case, got, want)


def test_smeter_helper_matches_oracle():
    """t41rx_smeter_dbm is host arithmetic (Display.cpp:959-981): no GPU needed."""
    lib = O.tier_b()
    rng = np.random.default_rng(3)
    for v in np.concatenate([10.0 ** rng.uniform(-6, 6, 200), [0.0, 1.0, 40.0]]).astype(np.float32):
        for gc, rf, rfall in ((-2.0, 1, 1), (3.5, 15, -10), (0.0, 7, 20)):
            a, b = rx.smeter_dbm(float(v), gc, rf, rfall), lib.t41o_smeter_dbm(float(v), gc, rf, rfall)
            assert a == b or (np.isnan(a) and np.isnan(b)) or (np.isinf(a) and a == b), (v, gc, rf, rfall, a, b)
    for dbm in np.concatenate([rng.uniform(-160, 0, 300), [-127.0, -73.0, -73.0 + 1e-4, -200.0, 50.0]]).astype(np.float32):
        assert rx.smeter_bar(float(dbm)) == lib.t41o_smeter_bar(float(dbm)), dbm
    assert rx.smeter_bar(-127.0) == 0 and rx.smeter_bar(-73.0) == 108 and rx.smeter_bar(0.0) == 180
    # the comment in the reference: audioMaxSquaredAve = 40 is about S9 (-73 dBm) on a calibrated band
    assert -80.0 < rx.smeter_dbm(40.0, -2.0, 1, 1) < -50.0


def test_wav_reader_matches_reference_golden(tmp_path):
    """t41rx_load_wav / t41rx_read_wave against what the reference's load_wav / readWave (Utility.cpp:773-888, run
    from its own translation unit by tests/golden/make_golden.py) returned for the same files: return codes, number
    of successful reads (the reference's quirky end test included), every sample."""
    import wav_cases
    golden = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_vectors.npz"))
    for name, (data, limit, chunk) in wav_cases.cases().items():
        p = tmp_path / (name + ".wav")
        if data is not None:
            p.write_bytes(data)
        state = {}

        def load(path, lim):
            state["w"] = rx.WavReader(path, lim)
            return state["w"].rc

        rc, n, full, tail = wav_cases.run(load, lambda k: state["w"].read(k), str(p), data, limit, chunk)
        state["w"].close()
        assert [rc, n] == list(golden["wav/%s/rc_n" % name]), name
        assert np.array_equal(full.view(np.uint32), golden["wav/%s/full" % name].view(np.uint32)), name
        assert np.array_equal(tail.view(np.uint32), golden["wav/%s/tail" % name].view(np.uint32)), name
    assert list(golden["wav/pcm16_fmt16_chunk128/rc_n"]) == [0, 39]      # 5000 samples = 39 reads of 128 + 8 samples the end test never delivers
    assert [int(golden["wav/%s/rc_n" % k][0]) for k in ("missing", "fmt20", "stereo", "too_long")] == [-1, -2, -3, -4]


@pytest.mark.skipif(not O.tier_a_available(), reason="oracle/_ref/libt41ref.so not built (needs /root/reference)")
def test_wav_reader_matches_reference_live(tmp_path):
    import wav_cases
    for name, (data, limit, chunk) in wav_cases.cases().items():
        p = tmp_path / (name + ".wav")
        if data is not None:
            p.write_bytes(data)
        ref = O.RefStream()
        want = wav_cases.run(ref.load_wav, ref.read_wave, str(p), data, limit, chunk)
        state = {}

        def load(path, lim):
            state["w"] = rx.WavReader(path, lim)
            return state["w"].rc

        got = wav_cases.run(load, lambda k: state["w"].read(k), str(p), data, limit, chunk)
        state["w"].close()
        assert got[:2] == want[:2], name
        assert np.array_equal(got[2], want[2]) and np.array_equal(got[3], want[3]), name


def test_bench_reference_arm_prints_one_json_line():
    """`bench.py --impl reference` (the CPU chain on the host cores: oracle/_ref when built, else the oracle port) must
    run without a GPU and print the contract's JSON line."""
    import json
    import subprocess
    import sys
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                          "--cpu-seconds", "1", "--blocks", "8"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["value"] > 0 and line["unit"] == "Msamples/s"
    assert line["cpu_baseline"]["kind"] in ("reference", "port") and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0


@pytest.mark.parametrize("S,T,budget,n_recv,n_blocks", [(64, 16, 2 ** 20, 7, 16), (4, 64, 2 ** 19, 1, 63)],
                         ids=["receivers_sampled", "blocks_sampled"])
def test_bench_dump_outputs_is_a_fixed_bounded_sample(tmp_path, monkeypatch, S, T, budget, n_recv, n_blocks):
    """`bench.py --dump-outputs`: float32 files within the byte budget; distinct receivers and blocks in increasing order,
    chosen by the shapes alone (the same ones for other output values); each dumped value taken unchanged from the
    step's output (waterfall words read as unsigned)."""
    import bench
    torch = pytest.importorskip("torch")
    monkeypatch.setattr(bench, "DUMP_BYTES", budget)
    # audio value = position in the output, so that every dumped sample names its receiver and block
    audio = torch.arange(S * T * 2048, dtype=torch.float32).reshape(S, T, 2048)
    spec = torch.arange(S * 512, dtype=torch.int32).reshape(S, 1, 512).to(torch.int16)
    wf = -1 - spec
    picked = []
    for d, offset in (("a", 0.0), ("b", 0.5)):
        bench.dump_outputs(str(tmp_path / d), audio + offset, spec, wf)
        files = sorted(os.listdir(tmp_path / d))
        assert files == ["audio.npy", "spec.npy", "wf.npy"]
        assert sum(os.path.getsize(tmp_path / d / f) for f in files) <= budget + 3 * 128
        out = {f[:-4]: np.load(tmp_path / d / f) for f in files}
        assert all(a.dtype == np.float32 for a in out.values())
        assert out["audio"].shape == (n_recv, n_blocks, 2048) and out["spec"].shape == out["wf"].shape == (n_recv, 1, 512)
        pos = np.floor(out["audio"][:, :, 0]).astype(np.int64) // 2048
        recv, blocks = pos[:, 0] // T, pos[0] % T
        assert np.array_equal(pos, recv[:, None] * T + blocks[None, :])
        assert np.all(np.diff(recv) > 0) and np.all(np.diff(blocks) > 0)
        assert np.array_equal(out["audio"], (audio + offset).numpy()[recv][:, blocks])
        assert np.array_equal(out["spec"], spec.numpy()[recv].astype(np.float32))
        assert np.array_equal(out["wf"], wf.numpy()[recv].view(np.uint16).astype(np.float32))
        picked.append((recv, blocks))
    assert all(np.array_equal(a, b) for a, b in zip(*picked))


def test_filter_set_slots_are_reused_in_a_tuning_sweep():
    """A long sweep of filter cut-offs on one receiver (HostModel::Apply re-uses the slot nobody references any more instead
    of growing the table, rx_host.cpp) must leave exactly the tables a fresh design of the last setting has (the AGC
    block keeps the sticky hang_thresh of its own history, B12: compared separately on equal AGC sequences)."""
    seq = [cases.P(mode=cases.USB, f_lo_cut=200 + 10 * k, f_hi_cut=2400 + 25 * k) for k in range(40)]
    seq += [cases.P(mode=cases.NFM, nfm_filter_bw=9000 + 500 * k) for k in range(6)]
    seq += [cases.P(mode=cases.LSB, f_lo_cut=-2900, f_hi_cut=-150)]
    swept = rx.design_tables([rx_driver.to_rx_params(p) for p in seq])
    fresh = rx.design_tables([rx_driver.to_rx_params(seq[-1])])
    for k in ("dec1", "dec2", "int1", "int2", "mask", "am_lp", "zoom_fir"):
        assert np.array_equal(np.asarray(swept[k]).view(np.uint32), np.asarray(fresh[k]).view(np.uint32)), k
    # NFM re-designs the decimators with its own cut-off (B15): the sweep went through NFM, the fresh receiver did not,
    # and both end on the LSB design: equal above means the re-used slots really were re-designed


def test_bench_workloads_are_valid_product_parameters():
    """bench.py builds C2 - C5 through the product's own C-ABI (no oracle library in the GPU arm): every parameter set must
    pass the library's validation, and the receiver counts / shapes are BASELINE.json's."""
    import bench
    for name, n in (("c2", 16), ("c3", 16), ("c4", 5), ("c5", 4)):
        params, sigs = bench.workload(2, name)
        assert len(params) == len(sigs) == n
        for p, s in zip(params, sigs):
            assert isinstance(p, rx.Params)
            rx.design_tables([p])                         # raises on an invalid parameter set
            assert s.shape == (2, 2048, 2) and s.dtype == np.float32
    assert bench.EXTRA_CONFIGS["c3"][0] == 8192 and bench.EXTRA_CONFIGS["c4"][0] == 16384 and bench.EXTRA_CONFIGS["c5"][0] == 32768
    assert {p.mode for p in bench.workload(2, "c3")[0]} == {3, 8}           # NFM + SAM
    assert sorted({p.spectrum_zoom for p in bench.workload(2, "c4")[0]}) == [0, 1, 2, 3, 4]
