#!/usr/bin/env python3
"""bench.py — throughput of the T41 receive-chain hot path on B200.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one pass of the fused RX chain (ProcessIQData x n_blocks) over the whole bank of
virtual receivers of a rank.  Workload = BASELINE.json configs[1]: 1024 concurrent receivers per
GPU, SSB + AM mixed, 192 kS/s, per-receiver NCO frequency, AGC on, one spectrum + waterfall
row per receiver per step.  With N > 1 (torchrun, one rank per GPU) every rank runs its own 1024
receivers (receivers are independent: no data-path collective; weak scaling) and the time is
the max over ranks.

Prints ONE JSON line (rank 0).  `value`  : complex Msamples/s, inputs resident in HBM, CUDA events.
                                 `e2e`    : same metric through t41rx_process with pinned HOST
                                            buffers (H2D + kernel + D2H inside the timed region).
                                 `roofline`: algorithmic bytes / measured kernel time vs measured HBM peak.
                                 `cpu_baseline`: the CPU oracle on the host cores, bounded sample.
`configs` : BASELINE.json configs[2..4] on the same GPUs, device-resident, each with its own roofline:
            c3 = 8192 receivers NFM + SAM with AGC 1-4 (8192 / N per GPU), c4 = 16384 receivers, zoom x1..x16,
            every block a spectrum + waterfall row (16384 / N per GPU), c5 = 32768 receivers PSK31 front end
            with the DBPSK + varicode tap (32768 / N per GPU).  `value` stays C2.
`--impl reference` times the reference's own CPU implementation of the path (oracle/_ref, the
reference translation units compiled in place; falls back to the oracle port) on all host cores.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

# dram__bytes_read.sum + dram__bytes_write.sum of one t41rx_stream_rx_kernel launch of this workload from the
# committed `ncu --set full` capture (profiles/summary_r02.md: 1078.8 MB read + 500.8 MB written at 1024
# receivers x 64 blocks; the algorithmic figure is 1610.6 MB, part of the last audio blocks is still in L2 at
# kernel end); only meaningful for the default workload, None otherwise
TRAFFIC_BYTES_PER_LAUNCH = 1078842000 + 500761344
# smsp__inst_executed.sum / stream-blocks of the same capture: warp-instructions the stream kernel executes per
# 2048-sample block of one receiver (profiles/summary_r02.md section 3)
WARP_INSTR_PER_STREAM_BLOCK = 7931
N_SMS, ISSUE_SLOTS_PER_SM = 148, 4

METRIC = "aggregate IQ Msamples/s (full RX chain)"
UNIT = "Msamples/s"
N_DISTINCT = 16


def positive_int(s):
    v = int(s)
    if v < 1:
        raise argparse.ArgumentTypeError("must be at least 1, got %d" % v)
    return v


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=positive_int, default=10, help="timed steps of every timed loop")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--streams", type=int, default=1024, help="virtual receivers per GPU")
    ap.add_argument("--blocks", type=int, default=64, help="2048-sample blocks per receiver per step")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="CPU work budget of the cpu_baseline sample")
    ap.add_argument("--rows-per-step", type=int, default=1, choices=[0, 1],
                    help="spectrum + waterfall rows per receiver per step (the first block of a step)")
    ap.add_argument("--gather-rows", action="store_true",
                    help="after the timed region, gather every rank's spectrum rows to rank 0 over NCCL (optional "
                         "path of SURVEY 8(e); reported as rows_gather_ms)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-q15", action="store_true", help="skip the device-resident q15 leg (value_q15)")
    ap.add_argument("--no-extra-configs", action="store_true", help="skip BASELINE.json configs[2..4] (c3 / c4 / c5)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned (audio, spectrum and waterfall rows of "
                         "a fixed sample of receivers) as DIR/<name>.npy in float32; with several GPUs, rank 0's "
                         "receivers only")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    return args


USB, LSB, AM, NFM, PSK31, SAM = 0, 1, 2, 3, 5, 8     # SDT.h:57-68 (t41rx.h T41RX_DEMOD_*)


def workload(n_blocks, name="c2"):
    """(params, signals) of a bank's N_DISTINCT-or-fewer distinct receivers; receiver s of a bank runs number
    s % len(params).  Parameters are built through the product's own C-ABI (rx.make_params): nothing under oracle/
    is touched here.
    c2: even receivers USB (+300..+3000), odd AM (+-3000), per-receiver tone / NCO (BASELINE.json configs[1]).
    c3: even NFM (+-2.5 kHz deviation), odd SAM (carrier offset U[-200, 200] Hz), AGC mode cycling 1..4, a -20 dB level
        step in the middle of the step (configs[2]).
    c4: zoom index = receiver % 5 (x1 .. x16), two tones + noise, every block a row (configs[3]).
    c5: PSK31 front end: +-100 Hz mask, AGC off, DBPSK + varicode tap on a carrier tuned to DC (configs[4])."""
    from t41_sdr_b200 import rx, synth
    P = rx.make_params
    r = np.random.Generator(np.random.PCG64(2024))
    params, sigs = [], []
    if name == "c2":
        for k in range(N_DISTINCT):
            nco = int(r.integers(-20000, 20001))
            if k % 2 == 0:
                params.append(P(mode=USB, f_lo_cut=300, f_hi_cut=3000, nco_freq=nco, agc_mode=1))
                sigs.append(synth.tone(900 + k, n_blocks, float(r.uniform(300, 2700)), mode=USB, nco_freq=nco))
            else:
                params.append(P(mode=AM, nco_freq=nco, agc_mode=1))
                sigs.append(synth.am(900 + k, n_blocks, mode=AM, nco_freq=nco, depth=0.5, f_mod=400.0))
    elif name == "c3":
        for k in range(N_DISTINCT):
            agc = 1 + (k % 4)
            if k % 2 == 0:
                params.append(P(mode=NFM, agc_mode=agc, nfm_filter_bw=12000))
                sigs.append(synth.nfm(300 + k, n_blocks, level_step_block=n_blocks // 2, level_step_db=-20.0))
            else:
                params.append(P(mode=SAM, agc_mode=agc))
                sigs.append(synth.am(300 + k, n_blocks, mode=SAM, carrier_offset=float(r.uniform(-200, 200)), depth=0.5,
                                     level_step_block=n_blocks // 2, level_step_db=-20.0))
    elif name == "c4":
        for z in range(5):
            params.append(P(mode=USB, spectrum_zoom=z, current_scale=1))
            sigs.append(synth.two_tone(40 + z, n_blocks, 46500.0, 50500.0))
    elif name == "c5":
        for k in range(4):
            params.append(P(mode=USB, f_lo_cut=-100, f_hi_cut=100, agc_mode=0, psk31_enable=1))
            sigs.append(synth.tone(50 + k, n_blocks, 0.0))
    else:
        raise ValueError(name)
    if name == "c2" and os.environ.get("T41RX_BENCH_WORKLOAD") == "c3":   # developer knob: C3 as the main line
        return workload(n_blocks, "c3")
    if os.environ.get("T41RX_BENCH_MODE"):       # developer knob: every receiver in one mode (0 USB, 2 AM) / AGC off (-1)
        m = int(os.environ["T41RX_BENCH_MODE"])
        for p in params:
            if m < 0:
                p.agc_mode = 0
            else:
                p.mode = m
                p.f_lo_cut, p.f_hi_cut = (300, 3000) if m == 0 else (-3000, 3000)
    if os.environ.get("T41RX_BENCH_EQ"):         # developer knob: receive equaliser on for every receiver (not the C2 metric)
        for p in params:
            p.receive_eq_flag = 1
            for i, v in enumerate([100, 80, 0, 120, 55, 100, 30, 90, 100, 10, 70, 100, 45, 100]):
                p.equalizer_rec[i] = v
    if os.environ.get("T41RX_BENCH_ZOOM"):       # developer knob (rows-kernel experiments)
        for p in params:
            p.spectrum_zoom = int(os.environ["T41RX_BENCH_ZOOM"])
    return params, sigs


def config_dict(args):
    return {"workload": "C2: %d concurrent virtual receivers per GPU, SSB+AM mixed, 192 kS/s, AGC Long, "
                        "per-receiver NCO, full RX chain fused" % args.streams,
            "receivers_per_gpu": args.streams, "blocks_per_step": args.blocks, "block_samples": 2048,
            "rows_per_receiver_per_step": args.rows_per_step, "distinct_waveforms": N_DISTINCT,
            "l2_policy": "inputs larger than L2 (%.0f MiB of I/Q per step per GPU)" % (
                args.streams * args.blocks * 16384 / 2 ** 20),
            "parallelism": "receivers sharded across GPUs, no data-path collective"}


# ---------------------------------------------------------------------------------------------
# CPU legs (the only places bench.py touches oracle/)
# ---------------------------------------------------------------------------------------------
def cpu_run(kind, params, sigs, n_blocks, seconds, cores):
    """Time the CPU chain on `cores` threads (ctypes releases the GIL).  Returns Msamples/s."""
    import oracle_py as O
    use_ref = (kind == "reference") and O.tier_a_available()
    if not use_ref and not os.path.exists(O.TIER_B_PATH):
        O.build_oracle()
    import ctypes as C

    def conv(p):                             # same field layout on both sides of the C-ABI (tests/rx_driver.py)
        q = O.Params()
        assert C.sizeof(q) == C.sizeof(p)
        C.memmove(C.byref(q), C.byref(p), C.sizeof(q))
        return q
    mk = (lambda p: O.RefStream(conv(p))) if use_ref else (lambda p: O.OracleStream(conv(p)))
    streams = [mk(params[i % len(params)]) for i in range(cores)]
    # calibrate on one thread
    t0 = time.perf_counter()
    streams[0].process(sigs[0][:min(n_blocks, 32)], 0)
    per_block = (time.perf_counter() - t0) / min(n_blocks, 32)
    reps = max(1, int(round(seconds / (per_block * n_blocks))))   # every thread runs ~`seconds` in parallel
    done = [0] * cores

    def work(i):
        sig = sigs[i % len(sigs)]
        for _ in range(reps):
            streams[i].process(sig, n_blocks)   # one spectrum row per pass, like the GPU step
            done[i] += n_blocks

    th = [threading.Thread(target=work, args=(i,)) for i in range(cores)]
    t0 = time.perf_counter()
    for t in th:
        t.start()
    for t in th:
        t.join()
    dt = time.perf_counter() - t0
    total_blocks = sum(done)
    return total_blocks * 2048 / dt / 1e6, ("reference" if use_ref else "port"), total_blocks, dt


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    params, sigs = workload(args.blocks)
    vals = []
    kind = "port"
    total = 0
    for _ in range(max(1, args.warmup)):
        cpu_run("reference", params, sigs, args.blocks, 1.0, cores)
    t_all0 = time.perf_counter()
    for _ in range(max(1, args.steps)):
        v, kind, blocks, dt = cpu_run("reference", params, sigs, args.blocks, max(1.0, args.cpu_seconds / max(1, args.steps)), cores)
        vals.append(v)
        total += blocks
    t_all = time.perf_counter() - t_all0
    value = statistics.median(vals)
    sample = "%d threads x private receivers, %d stream-blocks in %.1f s (C2 parameter mix)" % (cores, total, t_all)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_all / max(1, args.steps),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_dict(args),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    Q_OLD = Q.replace("clocks_event_reasons", "clocks_throttle_reasons")

    def __init__(self, device):
        self.device = device
        self.path = tempfile.mktemp(prefix="t41rx_clocks_", suffix=".csv")
        self.proc = None

    def start(self):
        try:
            q = self.Q
            probe = subprocess.run(["nvidia-smi", "-i", str(self.device), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                   capture_output=True, text=True, timeout=20)
            if probe.returncode != 0 or "not a valid" in (probe.stdout + probe.stderr).lower():
                q = self.Q_OLD
            self.fh = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "50"], stdout=self.fh,
                                         stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        try:
            self.proc.terminate()
            self.proc.wait(timeout=5)
            self.fh.close()
            sm, mx, pw, reasons = [], [], [], set()
            for ln in open(self.path):
                f = [x.strip() for x in ln.split(",")]
                if len(f) < 9:
                    continue
                try:
                    sm.append(float(f[1]))
                    mx.append(float(f[2]))
                    pw.append(float(f[3]))
                except ValueError:
                    continue
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            if sm:
                # "under load" = samples drawing more than half of the highest power seen
                busy = [c for c, p in zip(sm, pw) if p >= 0.5 * max(pw)] or sm
                out = {"sm_mhz": statistics.median(busy), "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                       "samples": len(sm), "power_w_max": max(pw)}
        except Exception:
            pass
        finally:
            try:
                os.unlink(self.path)
            except OSError:
                pass
        return out


def bind_to_gpu_numa_node(local):
    """Best effort: run this rank (and first-touch its pinned host buffers) on the NUMA node the GPU hangs off, so
    that N ranks do not all stage through node 0's memory.  Returns a short description for the JSON line."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(local)
        bdf = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bdf).read().strip())
        if node < 0:
            # no NUMA node in sysfs (a VM / container often hides it): ask NVML which CPUs are close to the GPU
            try:
                import pynvml
                pynvml.nvmlInit()
                h = pynvml.nvmlDeviceGetHandleByPciBusId(bdf.encode())
                words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
                ideal = {64 * i + b for i, w in enumerate(words) for b in range(64) if (int(w) >> b) & 1}
                allowed = os.sched_getaffinity(0)
                use = ideal & allowed
                if use and use != allowed:
                    os.sched_setaffinity(0, use)
                return {"numa_node": None, "source": "nvml", "gpu_local_cpus": len(ideal), "allowed_cpus": len(allowed),
                        "bound_to": len(use) if use else 0, "pci": bdf}
            except Exception as e:     # noqa: BLE001 - diagnostic only
                return {"numa_node": None, "note": "no NUMA node for %s in sysfs; NVML: %s: %s" % (bdf, type(e).__name__, e)}
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0) or cpus
        if cpus:
            os.sched_setaffinity(0, cpus)
        return {"numa_node": node, "cpus": len(cpus), "pci": bdf}
    except Exception as e:     # noqa: BLE001 - diagnostic only
        return {"numa_node": None, "note": "%s: %s" % (type(e).__name__, e)}


def measured_peak():
    try:
        pk = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(pk["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


# ---------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------
EXTRA_CONFIGS = {
    # name: (receivers over all GPUs, blocks per step, row_every, psk tap, algorithmic bytes per stream-block, text)
    "c3": (8192, 64, 0, False, 24576, "C3: 8192 receivers, even NFM / odd SAM, AGC modes 1-4, -20 dB level step mid-step"),
    "c4": (16384, 32, 1, False, 16384 + 2048, "C4: 16384 receivers, zoom x1..x16 by receiver, every block a spectrum + "
                                              "waterfall row (the audio chain runs beside it)"),
    "c5": (32768, 24, 0, True, 24576, "C5: 32768 receivers, PSK31 front end (+-100 Hz mask, AGC off) + DBPSK + varicode tap"),
}


# what --dump-outputs writes stays under 64 MB in all
DUMP_BYTES = 48 * 2 ** 20


def dump_outputs(out_dir, audio, spec, wf):
    """Write what one t41rx_process_device call returned to its caller - audio [S, T, 2048] float32 and, when the call
    made rows, spectrum rows [S, R, 512] int16 and waterfall rows [S, R, 512] uint16 - as float32 DIR/<name>.npy files:
    every receiver and block when that fits DUMP_BYTES, else a sample of receivers (and of blocks) drawn from a fixed
    seed.  The sample depends on the shapes only, so two builds run with the same arguments write comparable files."""
    S, T, B = audio.shape
    R = spec.shape[1] if spec is not None else 0
    r = np.random.Generator(np.random.PCG64(2024))
    nb = min(T, (DUMP_BYTES // 4 - 2 * R * 512) // B)
    nr = min(S, DUMP_BYTES // (4 * (nb * B + 2 * R * 512)))
    recv = np.sort(r.choice(S, nr, replace=False))
    blocks = np.sort(r.choice(T, nb, replace=False))
    out = {"audio": audio[recv][:, blocks].cpu().numpy()}
    if R:
        out["spec"] = spec[recv].cpu().numpy().astype(np.float32)
        out["wf"] = wf[recv].cpu().numpy().view(np.uint16).astype(np.float32)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_extra_config(name, world, local, dev, steps, peak):
    """One of BASELINE.json configs[2..4], device-resident, sharded over the ranks (strong scaling: the config
    fixes the receiver count).  Returns this rank's numbers; the caller reduces the time over ranks."""
    import torch
    from t41_sdr_b200 import rx
    S_all, T, row_every, psk, bytes_per_block, text = EXTRA_CONFIGS[name]
    S = S_all // world
    params, sigs = workload(T, name)
    D = len(params)
    base = torch.from_numpy(np.stack(sigs)).to(dev)
    iq = base.index_select(0, torch.arange(S, device=dev) % D).contiguous()
    del base
    R = (T + row_every - 1) // row_every if row_every else 0
    audio = torch.empty((S, T, 2048), dtype=torch.float32, device=dev)
    spec = torch.empty((S, max(R, 1), 512), dtype=torch.int16, device=dev)
    wf = torch.empty((S, max(R, 1), 512), dtype=torch.int16, device=dev)
    bits = torch.empty((S, T), dtype=torch.int8, device=dev) if psk else None
    chars = torch.empty((S, T), dtype=torch.uint8, device=dev) if psk else None
    stream = torch.cuda.Stream(device=dev)
    with rx.Receiver(S, device=local) as eng:
        eng.set_params_each([params[s % D] for s in range(S)])

        def step():
            eng.process_device(iq.data_ptr(), audio.data_ptr(), T, row_every, spec.data_ptr() if R else None,
                               wf.data_ptr() if R else None, bits.data_ptr() if psk else None,
                               chars.data_ptr() if psk else None, 0, stream.cuda_stream)
        for _ in range(3):
            step()
        torch.cuda.synchronize()
        l0 = eng.kernel_launches()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(steps):
            step()
        e1.record(stream)
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        launches = (eng.kernel_launches() - l0) // steps
        check = float(audio[::max(1, S // 7), -1, ::257].abs().double().sum().item())
    del iq, audio, spec, wf
    torch.cuda.empty_cache()
    return dict(name=name, text=text, S=S, S_all=S_all, T=T, R=R, ms=ms, bytes_per_block=bytes_per_block, launches=launches,
                check=check)


def extra_config_entry(r, ms_max, world, peak):
    blocks = r["S_all"] * r["T"]
    achieved = (r["S"] * r["T"] * r["bytes_per_block"]) / (ms_max * 1e-3) / 1e9      # per GPU
    e = {"workload": r["text"], "receivers": r["S_all"], "receivers_per_gpu": r["S"], "blocks_per_step": r["T"],
         "value": blocks * 2048 / (ms_max * 1e-3) / 1e6, "unit": UNIT, "ms_per_step": ms_max, "scaling": "strong",
         "kernel_launches_per_step": r["launches"],
         "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                      "algorithmic_bytes_per_stream_block": r["bytes_per_block"], "per": "GPU, all kernels of the step"},
         "checksum_audio": r["check"]}
    if r["R"]:
        e["rows_per_s"] = r["S_all"] * r["R"] / (ms_max * 1e-3)
    return e


def ours(args):
    import torch
    import torch.distributed as dist
    from t41_sdr_b200 import rx, sharding

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the RX chain has no CPU path (use --impl reference for the CPU chain)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)

    S, T = args.streams, args.blocks
    row_every = T if args.rows_per_step else 0
    params, sigs = workload(T)
    eng = rx.Receiver(S, device=local)
    eng.set_params_each([params[s % len(params)] for s in range(S)])

    # synthetic input resident in HBM: receiver s gets waveform s % N_DISTINCT
    base = torch.from_numpy(np.stack(sigs)).to(dev)                       # [D, T, 2048, 2]
    idx = torch.arange(S, device=dev) % len(sigs)
    iq = base.index_select(0, idx).contiguous()                            # [S, T, 2048, 2]
    del base
    audio = torch.empty((S, T, 2048), dtype=torch.float32, device=dev)
    spec = torch.empty((S, 1, 512), dtype=torch.int16, device=dev)
    wf = torch.empty((S, 1, 512), dtype=torch.int16, device=dev)
    stream = torch.cuda.Stream(device=dev)     # a real (non-default) stream: the kernel is launched on it
    torch.cuda.synchronize()

    dev_flags = int(os.environ.get("T41RX_BENCH_FLAGS", "0"))     # developer knob (t41rx_process flags; 0 = the metric)

    def step():
        eng.process_device(iq.data_ptr(), audio.data_ptr(), T, row_every, spec.data_ptr(), wf.data_ptr(),
                           None, None, dev_flags, stream.cuda_stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(3, args.warmup)):
        step()
    barrier()
    clocks = ClockSampler(local)
    clocks.start()
    for _ in range(3):          # give the sampler something to see before the short timed region
        step()
    launches0 = eng.kernel_launches()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    t_start = torch.cuda.Event(enable_timing=True)
    t_end = torch.cuda.Event(enable_timing=True)
    t_start.record(stream)
    for a, b in evs:
        a.record(stream)
        step()
        b.record(stream)
    t_end.record(stream)
    barrier()
    total_ms = t_start.elapsed_time(t_end)
    launch_ms = [a.elapsed_time(b) for a, b in evs]
    gpu_launches = eng.kernel_launches() - launches0
    if args.dump_outputs and rank == 0:         # before the q15 leg below writes the same rows
        dump_outputs(args.dump_outputs, audio, spec if row_every else None, wf if row_every else None)

    total_ms_max = sharding.max_over_ranks(total_ms, dev)
    samples_per_step = world * S * T * 2048
    value = samples_per_step * args.steps / (total_ms_max * 1e-3) / 1e6

    # roofline of the dominant kernel (t41rx_stream_rx_kernel: one launch per step, the whole chain except the
    # display spectrum of the row-producing block, which t41rx_rows_kernel does): CUDA events recorded by the
    # library on the launch stream around exactly that kernel, over the timed steps
    kernel_ms = eng.stream_kernel_times(min(args.steps, 32))
    kernel_name = "t41rx_stream_rx_kernel"
    if not kernel_ms:          # developer knobs can send every receiver to the bit-exact kernel (all SAM)
        kernel_ms, kernel_name = launch_ms, "t41rx_fused_rx_kernel"
    bytes_per_launch = S * T * rx.BYTES_PER_BLOCK
    avg_launch_s = statistics.mean(kernel_ms) * 1e-3
    achieved = bytes_per_launch / avg_launch_s / 1e9
    peak, peak_src = measured_peak()
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": TRAFFIC_BYTES_PER_LAUNCH if (S, T) == (1024, 64) else None, "kernel": kernel_name, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": bytes_per_launch, "avg_launch_ms": statistics.mean(kernel_ms),
                "step_ms_all_kernels": statistics.mean(launch_ms),
                "share_of_step": statistics.mean(kernel_ms) / statistics.mean(launch_ms)}

    # the same steps on the firmware's own q15 block format, device-resident (t41rx_process_device_q15: the chain
    # kernels convert at their loads and stores; 6 B of HBM traffic per complex sample instead of 12)
    value_q15 = None
    if not args.no_q15:
        iq16 = torch.round(iq * 32768.0).to(torch.int16)                  # the synthetic I/Q is q15 / 32768
        audio16 = torch.empty((S, T, 2048), dtype=torch.int16, device=dev)

        def step16():
            eng.process_device_q15(iq16.data_ptr(), audio16.data_ptr(), T, row_every, spec.data_ptr(), wf.data_ptr(),
                                   None, None, dev_flags, stream.cuda_stream)
        for _ in range(3):
            step16()
        barrier()
        q0, q1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        q0.record(stream)
        for _ in range(args.steps):
            step16()
        q1.record(stream)
        barrier()
        q_ms = sharding.max_over_ranks(q0.elapsed_time(q1), dev) / args.steps
        gpu_launches = eng.kernel_launches() - launches0
        kq = eng.stream_kernel_times(min(args.steps, 32))
        pk, _ = measured_peak()
        kq_ms = statistics.mean(kq) if kq else q_ms
        ach = S * T * rx.BYTES_PER_BLOCK_Q15 / (kq_ms * 1e-3) / 1e9
        value_q15 = {"value": samples_per_step / (q_ms * 1e-3) / 1e6, "unit": UNIT, "ms_per_step": q_ms,
                     "api": "t41rx_process_device_q15 (q15 I/Q in, q15 audio out, resident in HBM)",
                     "roofline": {"bound": "hbm", "achieved": ach, "peak": pk, "unit": "GB/s", "frac": ach / pk,
                                  "algorithmic_bytes_per_stream_block": rx.BYTES_PER_BLOCK_Q15,
                                  "kernel": "t41rx_stream_rx_q15_kernel", "avg_launch_ms": kq_ms},
                     "checksum_audio": float(audio16[::97, -1, ::31].abs().double().sum().item() / 32768.0)}
        del iq16, audio16

    # end to end through the host-buffer C-ABI calls, pinned host buffers, H2D + kernels + D2H inside the timed
    # region: `e2e` = t41rx_process_q15, the firmware's own block format (q15 I/Q in, q15 audio out, what the
    # codec queues of Process.cpp:102-111,936-937 carry); `e2e_float` = t41rx_process on float blocks
    e2e = None
    e2e_float = None
    if not args.no_e2e:
        n_rows = 1 if row_every else 0
        numa = bind_to_gpu_numa_node(local)
        iq_host = iq.cpu()
        h_iq = torch.empty((S, T, 2048, 2), dtype=torch.float32).pin_memory()
        h_iq.copy_(iq_host)
        h_iq16 = torch.empty((S, T, 2048, 2), dtype=torch.int16).pin_memory()
        h_iq16.copy_(torch.round(iq_host * 32768.0).to(torch.int16))       # the synthetic I/Q is q15 / 32768
        del iq_host

        def host_out(dtype):
            return dict(audio=torch.empty((S, T, 2048), dtype=dtype).pin_memory().numpy(),
                        spec=torch.empty((S, max(n_rows, 1), 512), dtype=torch.int16).pin_memory().numpy()[:, :n_rows],
                        wf=torch.empty((S, max(n_rows, 1), 512), dtype=torch.int16).pin_memory().numpy().view(np.uint16)[:, :n_rows],
                        psk_bits=None, psk_chars=None)

        def timed(call):
            for _ in range(2):
                call()
            barrier()
            t0 = time.perf_counter()
            for _ in range(args.steps):
                call()
            torch.cuda.synchronize()
            return sharding.max_over_ranks(time.perf_counter() - t0, dev)

        out16 = host_out(torch.int16)
        h_iq16_np = h_iq16.numpy()
        dt = timed(lambda: eng.process_q15(h_iq16_np, row_every=row_every, out=out16))
        e2e = {"value": samples_per_step * args.steps / dt / 1e6, "unit": UNIT,
               "h2d_bytes_per_step": S * T * 8192, "d2h_bytes_per_step": S * T * 4096 + S * rx.BYTES_PER_ROW * args.rows_per_step,
               "api": "t41rx_process_q15 (q15 I/Q in, q15 audio + rows out; pinned host buffers)",
               "timed_with": "host wall clock around the blocking call, max over ranks",
               "host_link_per_rank": {"h2d_gbs": S * T * 8192 * args.steps / dt / 1e9,
                                      "d2h_gbs": (S * T * 4096 + S * rx.BYTES_PER_ROW * args.rows_per_step) * args.steps / dt / 1e9,
                                      "pinned_buffers": numa,
                                      "note": "the ranks of one box share the host's memory and PCIe / C2C links: this, "
                                              "not the GPUs, bounds e2e at N > 1"},
               "checksum_audio": float(np.abs(out16["audio"][::97, -1, ::31].astype(np.float64)).sum() / 32768.0)}
        outf = host_out(torch.float32)
        h_iq_np = h_iq.numpy()
        dt = timed(lambda: eng.process(h_iq_np, row_every=row_every, out=outf))
        e2e_float = {"value": samples_per_step * args.steps / dt / 1e6, "unit": UNIT,
                     "h2d_bytes_per_step": S * T * 16384, "d2h_bytes_per_step": S * T * 8192 + S * rx.BYTES_PER_ROW * args.rows_per_step,
                     "api": "t41rx_process (float blocks; pinned host buffers)",
                     "checksum_audio": float(np.abs(outf["audio"][::97, -1, ::31]).sum())}
        gpu_launches = eng.kernel_launches() - launches0

    rows_gather_ms = None
    if args.gather_rows and row_every:
        barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        gathered = sharding.gather_rows(spec, world * S, dst=0)
        g1.record()
        torch.cuda.synchronize()
        rows_gather_ms = sharding.max_over_ranks(g0.elapsed_time(g1), dev)
        if rank == 0:
            assert tuple(gathered.shape) == (world * S, 1, 512)

    # BASELINE.json configs[2..4] on the same GPUs (device-resident; C2 above stays `value`)
    extra = {}
    if not args.no_extra_configs:
        del iq, audio, spec, wf
        torch.cuda.empty_cache()
        peak_gbs, _ = measured_peak()
        for name in ("c3", "c4", "c5"):
            barrier()
            r = run_extra_config(name, world, local, dev, args.steps, peak_gbs)
            ms_max = sharding.max_over_ranks(r["ms"], dev)
            extra[name] = extra_config_entry(r, ms_max, world, peak_gbs)
            gpu_launches += r["launches"] * args.steps

    clk = clocks.stop()
    # explanatory second roofline: share of the SMs' issue slots the stream kernel used (instruction count of the
    # committed ncu capture, this run's kernel time and SM clock)
    if clk.get("sm_mhz"):
        issued = WARP_INSTR_PER_STREAM_BLOCK * S * T / (statistics.mean(kernel_ms) * 1e-3)
        slots = N_SMS * ISSUE_SLOTS_PER_SM * clk["sm_mhz"] * 1e6
        roofline["issue_slots"] = {"bound": "fp32 issue", "achieved": issued / 1e12, "peak": slots / 1e12,
                                   "unit": "T warp-instr/s", "frac": issued / slots,
                                   "warp_instr_per_stream_block": WARP_INSTR_PER_STREAM_BLOCK}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        v, kind, blocks, dt = cpu_run("port", params, sigs, T, args.cpu_seconds, cores)
        cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": kind,
               "sample": "%d stream-blocks of the same C2 mix on %d threads in %.1f s" % (blocks, cores, dt)}
        # BASELINE.json configs[0]: one receiver on ONE host core (USB, 2.7 kHz filter: the first C2 receiver)
        v1, kind1, blocks1, dt1 = cpu_run("port", params[:1], sigs[:1], T, min(4.0, args.cpu_seconds / 3), 1)
        cpu["single_core"] = {"value": v1, "unit": UNIT, "cores": 1, "kind": kind1,
                              "sample": "C1: one USB receiver, %d stream-blocks on one thread in %.1f s" % (blocks1, dt1)}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": max(3, args.warmup), "ms_per_step": total_ms_max / args.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": config_dict(args), "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "e2e_float": e2e_float,
                "gpu_launches": int(gpu_launches), "clocks": clk}
        if value_q15 is not None:
            line["value_q15"] = value_q15
        if extra:
            line["configs"] = extra
        if rows_gather_ms is not None:
            line["rows_gather_ms"] = rows_gather_ms
        print(json.dumps(line), flush=True)
    eng.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse_args()
    if args.impl == "reference":
        reference_arm(args)
    else:
        ours(args)


if __name__ == "__main__":
    main()
